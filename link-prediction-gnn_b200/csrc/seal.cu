// seal.cu - SEAL (Zhang & Chen 2018) on the device: enclosing-subgraph extraction with DRNL labels, and the DGCNN pieces that
// have no kernel elsewhere (tanh into a column slice, SortPooling, bias + activation + max-pool, im2col, the one-hot input layer).
//
// Extraction runs one CTA per query (grid-stride over the queries) with a private slice of the workspace: a stamp per graph node
// (`mark`, the query's stamp once the node has been seen) and a node list K. For query q = (u, v):
//   layer 0 = {u, v}; layer t = the neighbours of layer t-1's kept nodes not seen before. Every neighbour is stamped with one
//   atomicExch; the thread that stamps it first appends it to K. A layer with more than `cap` nodes is sorted by
//   (hash_u32(seed, (index_base + q) << 32 | node), node) and cut to its first `cap`: the dropped nodes stay seen, as in the
//   SEAL authors' k_hop_subgraph. K is then sorted ascending (the local order).
//   Edges: every (a, b), a and b in K, b in N(a), except (u, v) and (v, u); b's local id is its position in K (binary search).
//   DRNL (fill pass): level-synchronous BFS over the subgraph's own rows from u without v and from v without u, then
//   z = 1 + min(du, dv) + (d/2)(d/2 + d%2 - 1), d = du + dv; z(u) = z(v) = 1, 0 where either distance is infinite.
// Sorting is a bitonic network in which every comparator puts the smaller key first, so the positions past the list's end act as
// +infinity and are never touched. The count and fill passes run the same node-set code; the results depend on the query
// (and index_base + q) alone, never on the CTA that ran it or the number of CTAs.
#include "common.cuh"

namespace twowl {

constexpr int kSealThreads = 256;
constexpr int kSealWarps = kSealThreads / 32;

__device__ __forceinline__ uint32_t seal_hash(uint64_t seed, int64_t q, int32_t node) {
  return hash_u32(seed, ((uint64_t)q << 32) | (uint32_t)node);
}

struct ByNode {
  __device__ __forceinline__ bool operator()(int32_t a, int32_t b) const { return a < b; }
};
struct ByHash {
  uint64_t seed;
  int64_t q;
  __device__ __forceinline__ bool operator()(int32_t a, int32_t b) const {
    const uint32_t ha = seal_hash(seed, q, a), hb = seal_hash(seed, q, b);
    return ha < hb || (ha == hb && a < b);
  }
};

// ascending sort of a[0, n) by the whole CTA (n uniform); ends in a barrier
template <class Less>
__device__ void block_sort(int32_t* a, int n, Less less) {
  int p = 1;
  while (p < n) p <<= 1;
  for (int k = 2; k <= p; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < (p >> 1); i += blockDim.x) {
        int lo, hi;
        if (j == (k >> 1)) {   // mirrored half-cleaner: offset t of a k-block against offset k-1-t
          const int blk = i / j, t = i - blk * j;
          lo = blk * k + t;
          hi = blk * k + k - 1 - t;
        } else {
          lo = (i / j) * 2 * j + (i % j);
          hi = lo + j;
        }
        if (hi < n) {
          const int32_t x = a[lo], y = a[hi];
          if (less(y, x)) a[lo] = y, a[hi] = x;
        }
      }
      __syncthreads();
    }
  }
  __syncthreads();
}

__device__ __forceinline__ int lower_bound_k(const int32_t* K, int n, int32_t x) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (K[mid] < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

struct SealQueryArgs {
  const int64_t* ptr;
  const int32_t* adj;
  int64_t N;
  const int64_t* u;
  int64_t s_u;
  const int64_t* v;
  int64_t s_v;
  int64_t Q, index_base;
  int hops, cap;
  uint64_t seed;
  int32_t* ws;
  int64_t per_block;   // int32 slots of one CTA's slice
};

// the node set of query q into K (ascending) -> its size. mark holds stamps; the caller passes a stamp unique to the query.
__device__ int seal_nodes(const SealQueryArgs& A, int64_t q, int32_t a, int32_t b, int32_t stamp, int32_t* mark, int32_t* K,
                          int* s_cnt) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    K[0] = a < b ? a : b;
    K[1] = a < b ? b : a;
    mark[a] = stamp;
    mark[b] = stamp;
  }
  __syncthreads();
  int f0 = 0, f1 = 2;
  for (int t = 1; t <= A.hops; ++t) {
    if (threadIdx.x == 0) *s_cnt = 0;
    __syncthreads();
    for (int i = f0 + warp; i < f1; i += kSealWarps) {
      const int32_t x = K[i];
      for (int64_t e = A.ptr[x] + lane, end = A.ptr[x + 1]; e < end; e += 32) {
        const int32_t y = __ldg(A.adj + e);
        if (atomicExch(mark + y, stamp) != stamp) K[f1 + atomicAdd(s_cnt, 1)] = y;
      }
    }
    __syncthreads();
    int c = *s_cnt;
    __syncthreads();
    if (A.cap > 0 && c > A.cap) {
      block_sort(K + f1, c, ByHash{A.seed, A.index_base + q});
      c = A.cap;
    }
    f0 = f1;
    f1 += c;
  }
  block_sort(K, f1, ByNode{});
  return f1;
}

__device__ __forceinline__ bool is_target(int32_t x, int32_t y, int32_t a, int32_t b) {
  return (x == a && y == b) || (x == b && y == a);
}

__device__ __forceinline__ bool query_ok(int64_t a, int64_t b, int64_t N) { return a >= 0 && a < N && b >= 0 && b < N && a != b; }

// count pass: nodes[q], edges[q] (0 for a refused query); info[0] += bad ids, info[1] += u == v
__global__ void __launch_bounds__(kSealThreads) k_seal_count(SealQueryArgs A, int64_t* __restrict__ n_nodes, int64_t* __restrict__ n_edges,
                                                             unsigned long long* __restrict__ info) {
  __shared__ int s_cnt;
  __shared__ unsigned long long s_edges;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t* mark = A.ws + (int64_t)blockIdx.x * A.per_block;
  int32_t* K = mark + A.N;
  for (int64_t q = blockIdx.x; q < A.Q; q += gridDim.x) {
    const int64_t a = A.u[q * A.s_u], b = A.v[q * A.s_v];
    if (!query_ok(a, b, A.N)) {
      if (threadIdx.x == 0) {
        n_nodes[q] = 0, n_edges[q] = 0;
        const int bad = !(a >= 0 && a < A.N) + !(b >= 0 && b < A.N);
        if (bad) atomicAdd(info, (unsigned long long)bad);
        else atomicAdd(info + 1, 1ull);
      }
      continue;
    }
    if (threadIdx.x == 0) s_edges = 0;
    const int n = seal_nodes(A, q, (int32_t)a, (int32_t)b, (int32_t)(q + 1), mark, K, &s_cnt);
    unsigned long long m = 0;
    for (int i = warp; i < n; i += kSealWarps) {
      const int32_t x = K[i];
      for (int64_t e = A.ptr[x] + lane, end = A.ptr[x + 1]; e < end; e += 32) {
        const int32_t y = __ldg(A.adj + e);
        const int j = lower_bound_k(K, n, y);
        m += (j < n && K[j] == y && !is_target(x, y, (int32_t)a, (int32_t)b));
      }
    }
    if (m) atomicAdd(&s_edges, m);
    __syncthreads();
    if (threadIdx.x == 0) n_nodes[q] = n, n_edges[q] = (int64_t)s_edges;
    __syncthreads();
  }
}

// exclusive scan of c[0, n) in place into c[0, n] by the CTA (c[n] = total); sm: kSealWarps + 1 slots. Ends in a barrier.
__device__ void block_scan_i32(int32_t* c, int n, int32_t* sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t carry = 0;
  for (int base = 0; base < n; base += kSealThreads) {
    const int i = base + threadIdx.x;
    const int32_t x = i < n ? c[i] : 0;
    int32_t inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += o;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
      int32_t s = 0;
      for (int w = 0; w < kSealWarps; ++w) {
        const int32_t t = sm[w];
        sm[w] = s;
        s += t;
      }
      sm[kSealWarps] = s;
    }
    __syncthreads();
    if (i < n) c[i] = carry + sm[warp] + inc - x;
    carry += sm[kSealWarps];
    __syncthreads();
  }
  if (threadIdx.x == 0) c[n] = carry;
  __syncthreads();
}

// fill pass: nodes, z and the block-diagonal edge list of every query (ids offset by node_ptr[q])
__global__ void __launch_bounds__(kSealThreads) k_seal_fill(SealQueryArgs A, const int64_t* __restrict__ node_ptr,
                                                            const int64_t* __restrict__ edge_ptr, int64_t E_total,
                                                            int64_t* __restrict__ nodes, int32_t* __restrict__ z,
                                                            int64_t* __restrict__ edges) {
  __shared__ int s_cnt;
  __shared__ int32_t s_scan[kSealWarps + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t* mark = A.ws + (int64_t)blockIdx.x * A.per_block;
  int32_t* K = mark + A.N;
  int32_t* roff = K + A.N;         // N + 1
  int32_t* du = roff + A.N + 1;
  int32_t* dv = du + A.N;
  for (int64_t q = blockIdx.x; q < A.Q; q += gridDim.x) {
    const int64_t a = A.u[q * A.s_u], b = A.v[q * A.s_v];
    if (!query_ok(a, b, A.N)) continue;
    // stamps -(q + 1): distinct from the count pass's q + 1 and from 0
    const int n = seal_nodes(A, q, (int32_t)a, (int32_t)b, (int32_t)(-(q + 1)), mark, K, &s_cnt);
    const int64_t nb = node_ptr[q], eb = edge_ptr[q];
    for (int i = threadIdx.x; i < n; i += kSealThreads) nodes[nb + i] = K[i], du[i] = -1, dv[i] = -1;
    // per-node kept-edge counts
    for (int i = warp; i < n; i += kSealWarps) {
      const int32_t x = K[i];
      int cnt = 0;
      for (int64_t e = A.ptr[x] + lane, end = A.ptr[x + 1]; e < end; e += 32) {
        const int32_t y = __ldg(A.adj + e);
        const int j = lower_bound_k(K, n, y);
        cnt += (j < n && K[j] == y && !is_target(x, y, (int32_t)a, (int32_t)b));
      }
      cnt = __reduce_add_sync(0xffffffffu, cnt);
      if (lane == 0) roff[i] = cnt;
    }
    __syncthreads();
    block_scan_i32(roff, n, s_scan);
    // the rows: each warp compacts its node's kept neighbours in adjacency (= local id) order
    for (int i = warp; i < n; i += kSealWarps) {
      const int32_t x = K[i];
      int64_t o = eb + roff[i];
      for (int64_t e0 = A.ptr[x], end = A.ptr[x + 1]; e0 < end; e0 += 32) {
        const int64_t e = e0 + lane;
        int j = -1;
        if (e < end) {
          const int32_t y = __ldg(A.adj + e);
          const int p = lower_bound_k(K, n, y);
          if (p < n && K[p] == y && !is_target(x, y, (int32_t)a, (int32_t)b)) j = p;
        }
        const unsigned keep = __ballot_sync(0xffffffffu, j >= 0);
        if (j >= 0) {
          const int64_t w = o + __popc(keep & ((1u << lane) - 1u));
          edges[w] = nb + i;
          edges[E_total + w] = nb + j;
        }
        o += __popc(keep);
      }
    }
    __syncthreads();
    // DRNL: both BFS level by level over the subgraph's rows (col = edges[E_total + .] - nb)
    const int la = lower_bound_k(K, n, (int32_t)a), lb = lower_bound_k(K, n, (int32_t)b);
    if (threadIdx.x == 0) du[la] = 0, dv[lb] = 0;
    __syncthreads();
    for (int t = 0;; ++t) {
      int changed = 0;
      for (int i = threadIdx.x; i < n; i += kSealThreads) {
        const bool fu = du[i] == t, fv = dv[i] == t;
        if (!fu && !fv) continue;
        for (int64_t e = eb + roff[i], end = eb + roff[i + 1]; e < end; ++e) {
          const int j = (int)(edges[E_total + e] - nb);
          if (fu && j != lb && du[j] < 0) du[j] = t + 1, changed = 1;
          if (fv && j != la && dv[j] < 0) dv[j] = t + 1, changed = 1;
        }
      }
      if (!__syncthreads_or(changed)) break;
    }
    for (int i = threadIdx.x; i < n; i += kSealThreads) {
      int32_t lab;
      if (i == la || i == lb) {
        lab = 1;
      } else if (du[i] < 0 || dv[i] < 0) {
        lab = 0;
      } else {
        const int32_t d = du[i] + dv[i], h = d / 2;
        lab = 1 + (du[i] < dv[i] ? du[i] : dv[i]) + h * (h + d % 2 - 1);
      }
      z[nb + i] = lab;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- DGCNN pieces ------------------------------------------
constexpr int kElemThreads = 256;

// out[m, c] (+)= W[c * ld + min(z[m], ld - 1)]: the linear map of one_hot(z) by W [C, ld]
__global__ void __launch_bounds__(kElemThreads) k_label_gather(const float* __restrict__ W, int C, int64_t ld, const int64_t* __restrict__ z,
                                                               int64_t M, int accumulate, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / C;
    const int c = (int)(i - m * C);
    int64_t l = z[m];
    l = l < 0 ? 0 : (l >= ld ? ld - 1 : l);
    const float w = __ldg(W + (int64_t)c * ld + l);
    out[i] = accumulate ? out[i] + w : w;
  }
}

__global__ void __launch_bounds__(kElemThreads) k_tanh_slice_fwd(const float* __restrict__ h, int64_t M, int C, float* __restrict__ out,
                                                                 int64_t ld, int64_t off) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / C;
    out[m * ld + off + (i - m * C)] = tanhf(h[i]);
  }
}

__global__ void __launch_bounds__(kElemThreads) k_tanh_slice_bwd(const float* __restrict__ g, const float* __restrict__ y, int64_t ld,
                                                                 int64_t off, int64_t M, int C, float* __restrict__ dh) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / C, o = m * ld + off + (i - m * C);
    const float t = y[o];
    dh[i] = g[o] * (1.f - t * t);
  }
}

// one CTA per graph b (rows [gptr[b], gptr[b+1]) of X [*, D]): row i's rank = #rows with a larger key, or an equal key and a smaller
// index. Ranks below k are written: idx[b, rank] = i, out[b, rank] = X[i]; slots past the graph's size get -1 and zeros.
__global__ void __launch_bounds__(kElemThreads) k_sortpool_fwd(const float* __restrict__ X, int D, int key_col, const int64_t* __restrict__ gptr,
                                                               int64_t B, int k, float* __restrict__ out, int32_t* __restrict__ idx) {
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    const int64_t r0 = gptr[b];
    const int n = (int)(gptr[b + 1] - r0);
    for (int t = threadIdx.x; t < k; t += blockDim.x) idx[b * k + t] = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const float ki = X[(r0 + i) * D + key_col];
      int rank = 0;
      for (int j = 0; j < n && rank < k; ++j) {
        const float kj = X[(r0 + j) * D + key_col];
        rank += (kj > ki) || (kj == ki && j < i);
      }
      if (rank < k) idx[b * k + rank] = (int32_t)(r0 + i);
    }
    __syncthreads();
    for (int64_t e = threadIdx.x; e < (int64_t)k * D; e += blockDim.x) {
      const int t = (int)(e / D), c = (int)(e - (int64_t)t * D);
      const int32_t r = idx[b * k + t];
      out[(b * k + t) * D + c] = r >= 0 ? X[(int64_t)r * D + c] : 0.f;
    }
    __syncthreads();
  }
}

// dX[idx[s]] = g[s] for every kept slot s; every other row of dX 0 (a row is kept at most once: no accumulation)
__global__ void __launch_bounds__(kElemThreads) k_sortpool_bwd(const float* __restrict__ g, const int32_t* __restrict__ idx, int64_t S, int D,
                                                               float* __restrict__ dX) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < S * D; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / D;
    const int32_t r = idx[s];
    if (r >= 0) dX[(int64_t)r * D + (e - s * D)] = g[e];
  }
}

__device__ __forceinline__ float act_of(float x, int relu) { return relu ? fmaxf(x, 0.f) : x; }

// out[b, l, c] = drop(max_{s < pool} act(Y[b, l pool + s, c] + bias[c])), l < Lin / pool; the first maximum wins
__global__ void __launch_bounds__(kElemThreads) k_bias_act_fwd(const float* __restrict__ Y, const float* __restrict__ bias, int64_t B, int Lin,
                                                               int C, int pool, int relu, uint32_t thresh, float inv_keep, uint64_t seed,
                                                               float* __restrict__ out) {
  const int Lout = Lin / pool;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B * Lout * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bl = i / C;
    const int c = (int)(i - bl * C);
    const int64_t b = bl / Lout, l = bl - b * Lout;
    const float bc = bias[c];
    float m = act_of(Y[((b * Lin) + l * pool) * C + c] + bc, relu);
    for (int s = 1; s < pool; ++s) {
      const float x = act_of(Y[((b * Lin) + l * pool + s) * C + c] + bc, relu);
      if (x > m) m = x;
    }
    out[i] = thresh ? m * drop_scale(seed, (uint64_t)i, thresh, inv_keep) : m;
  }
}

__global__ void __launch_bounds__(kElemThreads) k_bias_act_bwd(const float* __restrict__ g, const float* __restrict__ Y, const float* __restrict__ bias,
                                                               int64_t B, int Lin, int C, int pool, int relu, uint32_t thresh, float inv_keep,
                                                               uint64_t seed, float* __restrict__ dY) {
  const int Lout = Lin / pool;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B * Lin * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bl = i / C;
    const int c = (int)(i - bl * C);
    const int64_t b = bl / Lin;
    const int l = (int)(bl - b * Lin), lo = l / pool;
    float d = 0.f;
    if (lo < Lout) {
      const float bc = bias[c];
      int arg = 0;
      float m = act_of(Y[((b * Lin) + lo * pool) * C + c] + bc, relu);
      for (int s = 1; s < pool; ++s) {
        const float x = act_of(Y[((b * Lin) + lo * pool + s) * C + c] + bc, relu);
        if (x > m) m = x, arg = s;
      }
      const float pre = Y[i] + bc;
      if (arg == l - lo * pool && (!relu || pre > 0.f)) {
        const int64_t o = (b * Lout + lo) * C + c;
        d = thresh ? g[o] * drop_scale(seed, (uint64_t)o, thresh, inv_keep) : g[o];
      }
    }
    dY[i] = d;
  }
}

// out[b L2 + p, c kw + j] = P[b, p + j, c], L2 = L1 - kw + 1
__global__ void __launch_bounds__(kElemThreads) k_im2col_fwd(const float* __restrict__ P, int64_t B, int L1, int C, int kw,
                                                             float* __restrict__ out) {
  const int L2 = L1 - kw + 1, W = C * kw;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B * L2 * W; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / W;
    const int col = (int)(i - row * W), c = col / kw, j = col - c * kw;
    const int64_t b = row / L2;
    const int p = (int)(row - b * L2);
    out[i] = P[(b * L1 + p + j) * C + c];
  }
}

// dP[b, t, c] = sum over j < kw (ascending) with 0 <= t - j < L2 of g[b L2 + t - j, c kw + j]
__global__ void __launch_bounds__(kElemThreads) k_im2col_bwd(const float* __restrict__ g, int64_t B, int L1, int C, int kw,
                                                             float* __restrict__ dP) {
  const int L2 = L1 - kw + 1, W = C * kw;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < B * L1 * C; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bt = i / C;
    const int c = (int)(i - bt * C);
    const int64_t b = bt / L1;
    const int t = (int)(bt - b * L1);
    float s = 0.f;
    for (int j = 0; j < kw; ++j) {
      const int p = t - j;
      if (p >= 0 && p < L2) s += g[(b * L2 + p) * W + c * kw + j];
    }
    dP[i] = s;
  }
}

}  // namespace twowl

using namespace twowl;

static int64_t seal_per_block(int64_t N) { return (int64_t)align_up((size_t)(5 * N + 1) * sizeof(int32_t)) / (int64_t)sizeof(int32_t); }

extern "C" size_t twowl_seal_workspace_bytes(int64_t num_nodes, int64_t Q, int64_t blocks) {
  if (num_nodes < 0 || Q < 0 || blocks < 1) return 0;
  return (size_t)blocks * (size_t)seal_per_block(num_nodes) * sizeof(int32_t) + align_up(scan_workspace_bytes(Q > 0 ? Q : 1));
}

static int seal_args(SealQueryArgs& A, const int64_t* ptr, const int32_t* adj, int64_t N, const int64_t* u, int64_t s_u, const int64_t* v,
                     int64_t s_v, int64_t Q, int64_t index_base, int32_t hops, int32_t cap, uint64_t seed, int64_t blocks, void* ws,
                     size_t ws_bytes, const char* op) {
  TW_CHECK_ARG(Q >= 0 && Q < 0x7fffffffLL && N >= 0 && N < 0x7fffffffLL && index_base >= 0 && index_base < (1LL << 31) &&
                   blocks >= 1 && blocks <= (1 << 20),
               "%s: bad sizes (0 <= Q < 2^31 - 1, 0 <= num_nodes < 2^31 - 1, 0 <= index_base < 2^31, 1 <= blocks <= 2^20)", op);
  TW_CHECK_ARG(hops >= 1 && hops <= 3, "%s: hops must be 1, 2 or 3", op);
  TW_CHECK_ARG(cap >= 0, "%s: max_nodes_per_hop must be >= 0", op);
  TW_CHECK_ARG(ptr && ws && (Q == 0 || (u && v)), "%s: null pointer", op);   // adj: NULL when nnz = 0
  TW_CHECK_WS(ws_bytes, twowl_seal_workspace_bytes(N, Q, blocks));
  A = SealQueryArgs{ptr, adj, N, u, s_u, v, s_v, Q, index_base, hops, cap, seed, static_cast<int32_t*>(ws), seal_per_block(N)};
  return 0;
}

extern "C" int twowl_seal_count(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* u, int64_t s_u, const int64_t* v,
                                int64_t s_v, int64_t Q, int64_t index_base, int32_t hops, int32_t max_nodes_per_hop, uint64_t seed,
                                int64_t blocks, int64_t* node_ptr, int64_t* edge_ptr, int64_t* info, void* ws, size_t ws_bytes, void* stream) {
  SealQueryArgs A;
  if (int rc = seal_args(A, ptr, adj, num_nodes, u, s_u, v, s_v, Q, index_base, hops, max_nodes_per_hop, seed, blocks, ws, ws_bytes,
                         "seal_count"))
    return rc;
  TW_CHECK_ARG(node_ptr && edge_ptr && info, "seal_count: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(info, 0, 2 * sizeof(int64_t), s));
  const int grid = (int)(Q < blocks ? (Q > 0 ? Q : 1) : blocks);
  void* sws = static_cast<char*>(ws) + (size_t)blocks * (size_t)A.per_block * sizeof(int32_t);
  if (Q > 0) {
    if (num_nodes > 0)
      TW_CUDA(cudaMemset2DAsync(A.ws, (size_t)A.per_block * sizeof(int32_t), 0, (size_t)num_nodes * sizeof(int32_t), grid, s));
    k_seal_count<<<grid, kSealThreads, 0, s>>>(A, node_ptr, edge_ptr, reinterpret_cast<unsigned long long*>(info));
    TW_LAUNCH_CHECK();
  }
  if (int rc = scan_exclusive_i64(node_ptr, node_ptr, Q, sws, s)) return rc;
  if (int rc = scan_exclusive_i64(edge_ptr, edge_ptr, Q, sws, s)) return rc;
  return 0;
}

extern "C" int twowl_seal_fill(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* u, int64_t s_u, const int64_t* v,
                               int64_t s_v, int64_t Q, int64_t index_base, int32_t hops, int32_t max_nodes_per_hop, uint64_t seed,
                               int64_t blocks, const int64_t* node_ptr, const int64_t* edge_ptr, int64_t n_edges, int64_t* nodes,
                               int32_t* z, int64_t* edge_index, void* ws, size_t ws_bytes, void* stream) {
  SealQueryArgs A;
  if (int rc = seal_args(A, ptr, adj, num_nodes, u, s_u, v, s_v, Q, index_base, hops, max_nodes_per_hop, seed, blocks, ws, ws_bytes,
                         "seal_fill"))
    return rc;
  TW_CHECK_ARG(n_edges >= 0, "seal_fill: bad sizes (n_edges >= 0)");
  TW_CHECK_ARG(node_ptr && edge_ptr && (Q == 0 || (nodes && z)) && (n_edges == 0 || edge_index), "seal_fill: null pointer");
  if (Q == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = (int)(Q < blocks ? Q : blocks);
  if (num_nodes > 0) TW_CUDA(cudaMemset2DAsync(A.ws, (size_t)A.per_block * sizeof(int32_t), 0, (size_t)num_nodes * sizeof(int32_t), grid, s));
  k_seal_fill<<<grid, kSealThreads, 0, s>>>(A, node_ptr, edge_ptr, n_edges, nodes, z, edge_index);
  TW_LAUNCH_CHECK();
  return 0;
}

static int elem_grid(int64_t n) { return grid_for(n, kElemThreads); }

extern "C" int twowl_label_gather(const float* W, int32_t C, int64_t ld, const int64_t* z, int64_t M, int32_t accumulate, float* out,
                                  void* stream) {
  TW_CHECK_ARG(C >= 1 && ld >= 1 && M >= 0, "label_gather: bad sizes (C >= 1, ld >= 1, M >= 0)");
  TW_CHECK_ARG(W && (M == 0 || (z && out)), "label_gather: null pointer");
  if (M == 0) return 0;
  k_label_gather<<<elem_grid(M * C), kElemThreads, 0, (cudaStream_t)stream>>>(W, C, ld, z, M, accumulate, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_tanh_slice_fwd(const float* h, int64_t M, int32_t C, float* out, int64_t ld, int64_t off, void* stream) {
  TW_CHECK_ARG(M >= 0 && C >= 1 && off >= 0 && off + C <= ld, "tanh_slice_fwd: bad sizes (M >= 0, C >= 1, 0 <= off, off + C <= ld)");
  TW_CHECK_ARG(M == 0 || (h && out), "tanh_slice_fwd: null pointer");
  if (M == 0) return 0;
  k_tanh_slice_fwd<<<elem_grid(M * C), kElemThreads, 0, (cudaStream_t)stream>>>(h, M, C, out, ld, off);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_tanh_slice_bwd(const float* g, const float* y, int64_t ld, int64_t off, int64_t M, int32_t C, float* dh, void* stream) {
  TW_CHECK_ARG(M >= 0 && C >= 1 && off >= 0 && off + C <= ld, "tanh_slice_bwd: bad sizes (M >= 0, C >= 1, 0 <= off, off + C <= ld)");
  TW_CHECK_ARG(M == 0 || (g && y && dh), "tanh_slice_bwd: null pointer");
  if (M == 0) return 0;
  k_tanh_slice_bwd<<<elem_grid(M * C), kElemThreads, 0, (cudaStream_t)stream>>>(g, y, ld, off, M, C, dh);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_sortpool_fwd(const float* X, int32_t D, int32_t key_col, const int64_t* gptr, int64_t B, int32_t k, float* out,
                                  int32_t* idx, void* stream) {
  TW_CHECK_ARG(D >= 1 && key_col >= 0 && key_col < D && B >= 0 && k >= 1 && B * k < 0x7fffffffLL,
               "sortpool_fwd: bad sizes (0 <= key_col < D, B >= 0, k >= 1, B k < 2^31)");
  TW_CHECK_ARG(gptr && (B == 0 || (X && out && idx)), "sortpool_fwd: null pointer");
  if (B == 0) return 0;
  k_sortpool_fwd<<<grid_for(B, 1), kElemThreads, 0, (cudaStream_t)stream>>>(X, D, key_col, gptr, B, k, out, idx);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_sortpool_bwd(const float* g, const int32_t* idx, int64_t B, int32_t k, int32_t D, int64_t n_rows, float* dX, void* stream) {
  TW_CHECK_ARG(D >= 1 && B >= 0 && k >= 1 && n_rows >= 0, "sortpool_bwd: bad sizes (D >= 1, B >= 0, k >= 1, n_rows >= 0)");
  TW_CHECK_ARG((n_rows == 0 || dX) && (B == 0 || (g && idx)), "sortpool_bwd: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  if (n_rows) TW_CUDA(cudaMemsetAsync(dX, 0, (size_t)n_rows * D * sizeof(float), s));
  if (B == 0) return 0;
  k_sortpool_bwd<<<elem_grid(B * k * D), kElemThreads, 0, s>>>(g, idx, B * k, D, dX);
  TW_LAUNCH_CHECK();
  return 0;
}

static int bias_act_check(int64_t B, int32_t Lin, int32_t C, int32_t pool, float p_drop, const char* op) {
  TW_CHECK_ARG(B >= 0 && Lin >= 1 && C >= 1 && (pool == 1 || pool == 2), "%s: bad sizes (B >= 0, Lin >= 1, C >= 1, pool 1 or 2)", op);
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "%s: p_drop must be in [0, 1)", op);
  return 0;
}

extern "C" int twowl_bias_act_fwd(const float* Y, const float* bias, int64_t B, int32_t Lin, int32_t C, int32_t pool, int32_t relu,
                                  float p_drop, uint64_t seed, float* out, void* stream) {
  if (int rc = bias_act_check(B, Lin, C, pool, p_drop, "bias_act_fwd")) return rc;
  TW_CHECK_ARG(bias && (B == 0 || (Y && out)), "bias_act_fwd: null pointer");
  const int64_t n = B * (Lin / pool) * C;
  if (n == 0) return 0;
  k_bias_act_fwd<<<elem_grid(n), kElemThreads, 0, (cudaStream_t)stream>>>(Y, bias, B, Lin, C, pool, relu, drop_thresh(p_drop),
                                                                          1.f / (1.f - p_drop), seed, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_bias_act_bwd(const float* g, const float* Y, const float* bias, int64_t B, int32_t Lin, int32_t C, int32_t pool,
                                  int32_t relu, float p_drop, uint64_t seed, float* dY, void* stream) {
  if (int rc = bias_act_check(B, Lin, C, pool, p_drop, "bias_act_bwd")) return rc;
  TW_CHECK_ARG(bias && (B == 0 || (g && Y && dY)), "bias_act_bwd: null pointer");
  if (B == 0) return 0;
  k_bias_act_bwd<<<elem_grid(B * Lin * C), kElemThreads, 0, (cudaStream_t)stream>>>(g, Y, bias, B, Lin, C, pool, relu, drop_thresh(p_drop),
                                                                                    1.f / (1.f - p_drop), seed, dY);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_im2col_fwd(const float* P, int64_t B, int32_t L1, int32_t C, int32_t kw, float* out, void* stream) {
  TW_CHECK_ARG(B >= 0 && C >= 1 && kw >= 1 && L1 >= kw, "im2col_fwd: bad sizes (B >= 0, C >= 1, 1 <= kw <= L1)");
  TW_CHECK_ARG(B == 0 || (P && out), "im2col_fwd: null pointer");
  if (B == 0) return 0;
  k_im2col_fwd<<<elem_grid(B * (L1 - kw + 1) * C * kw), kElemThreads, 0, (cudaStream_t)stream>>>(P, B, L1, C, kw, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_im2col_bwd(const float* g, int64_t B, int32_t L1, int32_t C, int32_t kw, float* dP, void* stream) {
  TW_CHECK_ARG(B >= 0 && C >= 1 && kw >= 1 && L1 >= kw, "im2col_bwd: bad sizes (B >= 0, C >= 1, 1 <= kw <= L1)");
  TW_CHECK_ARG(B == 0 || (g && dP), "im2col_bwd: null pointer");
  if (B == 0) return 0;
  k_im2col_bwd<<<elem_grid(B * L1 * C), kElemThreads, 0, (cudaStream_t)stream>>>(g, B, L1, C, kw, dP);
  TW_LAUNCH_CHECK();
  return 0;
}
