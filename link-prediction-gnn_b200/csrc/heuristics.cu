// heuristics.cu - neighbourhood link-prediction heuristics: common neighbours, Jaccard, Adamic-Adar, resource allocation.
//
// The graph is read as an undirected simple graph: N(x) = {y != x : (x, y) or (y, x) is an edge}, d(x) = |N(x)|.
//
// twowl_simple_adjacency builds it as a CSR whose rows are sorted and free of duplicates and self loops: both directions of
// every edge are keyed (row, neighbour) with dropped entries (self loops, bad ids) given the sentinel row N, then sorted with
// the library's stable LSD radix sort - by neighbour, then by row - and adjacent duplicates are compacted out by an exclusive
// scan of keep flags. Row starts come from a binary search of each row id in the sorted rows.
//
// twowl_link_heuristics intersects N(u) and N(v) for each query pair. The shorter list (ties: the smaller id) is probed
// into the longer one by binary search, so the work, and every floating-point sum, depends on the unordered pair only:
// score(u, v) and score(v, u) have the same bits. A pair with at most TWOWL_HEUR_LONG probes is handled by one 8-lane group.
// A longer one (two hubs) is cut into chunks of TWOWL_HEUR_CHUNK probes, one warp each; a chunk finds its range in the
// longer list by binary search (merge path) and writes an integer count and two double partials, which the pair's group
// then adds in chunk order. No floating-point atomics: two runs give the same bits.
#include "common.cuh"

namespace twowl {

constexpr int kHeurThreads = 256;
constexpr int kHeurGroup = 8;                                 // lanes per short pair
constexpr int kHeurGroups = kHeurThreads / kHeurGroup;        // short pairs per CTA pass
constexpr int kHeurWarps = kHeurThreads / 32;
constexpr int kHeurLong = TWOWL_HEUR_LONG;
constexpr int kHeurChunk = TWOWL_HEUR_CHUNK;

static int bits_for_value(int64_t max_value) {
  int b = 1;
  while (b < 32 && ((int64_t)1 << b) <= max_value) ++b;
  return b;
}

__device__ __forceinline__ int warp_sum_i(int v) { return __reduce_add_sync(0xffffffffu, v); }

// ---------------------------------------------------------------- simple adjacency -----------------
// entry i < E is (row[i], col[i]), entry E + i its reverse; key = neighbour, value = row (N for a dropped entry)
__global__ void __launch_bounds__(kHeurThreads) k_adj_keys(const int64_t* __restrict__ row, int64_t s_row, const int64_t* __restrict__ col,
                                                           int64_t s_col, int64_t E, int64_t N, uint32_t* __restrict__ nbr,
                                                           uint32_t* __restrict__ rws, int32_t* __restrict__ bad) {
  int nbad = 0;
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i - lane < E; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < E) {
      const int64_t r = row[i * s_row], c = col[i * s_col];
      const bool okr = r >= 0 && r < N, okc = c >= 0 && c < N;
      nbad += !okr + !okc;
      const bool keep = okr && okc && r != c;
      nbr[i] = keep ? (uint32_t)c : 0u;
      rws[i] = keep ? (uint32_t)r : (uint32_t)N;
      nbr[E + i] = keep ? (uint32_t)r : 0u;
      rws[E + i] = keep ? (uint32_t)c : (uint32_t)N;
    }
  }
  nbad = warp_sum_i(nbad);
  if (lane == 0 && nbad) atomicAdd(bad, nbad);
}

__device__ __forceinline__ bool adj_keep(const uint32_t* __restrict__ rws, const uint32_t* __restrict__ nbr, int64_t i, uint32_t N) {
  const uint32_t r = rws[i];
  return r < N && (i == 0 || r != rws[i - 1] || nbr[i] != nbr[i - 1]);
}

__global__ void __launch_bounds__(kHeurThreads) k_adj_flags(const uint32_t* __restrict__ rws, const uint32_t* __restrict__ nbr, int64_t M,
                                                            uint32_t N, int64_t* __restrict__ flag) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x)
    flag[i] = adj_keep(rws, nbr, i, N);
}

__global__ void __launch_bounds__(kHeurThreads) k_adj_fill(const uint32_t* __restrict__ rws, const uint32_t* __restrict__ nbr, int64_t M,
                                                           uint32_t N, const int64_t* __restrict__ pos, int32_t* __restrict__ adj) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x)
    if (adj_keep(rws, nbr, i, N)) adj[pos[i]] = (int32_t)nbr[i];
}

// ptr[r] = pos[first sorted entry with row >= r], r in [0, N]: empty rows and ptr[N] = nnz included
__global__ void __launch_bounds__(kHeurThreads) k_adj_ptr(const uint32_t* __restrict__ rws, int64_t M, int64_t N,
                                                          const int64_t* __restrict__ pos, int64_t* __restrict__ ptr) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= N; r += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = M;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if ((int64_t)rws[mid] < r)
        lo = mid + 1;
      else
        hi = mid;
    }
    ptr[r] = pos[lo];
  }
}

// ---------------------------------------------------------------- link heuristics -------------------
struct PairLists {
  const int32_t* S;   // shorter list (probed)
  const int32_t* L;   // longer list (searched)
  int ds, dl;
};

// the decomposition depends on the unordered pair only: shorter list first, ties by node id
__device__ __forceinline__ PairLists pair_lists(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t a, int64_t b,
                                                int64_t* da_out, int64_t* db_out) {
  const int64_t pa = ptr[a], pb = ptr[b];
  const int64_t da = ptr[a + 1] - pa, db = ptr[b + 1] - pb;
  *da_out = da, *db_out = db;
  const bool a_first = da < db || (da == db && a <= b);
  PairLists p;
  p.S = adj + (a_first ? pa : pb);
  p.L = adj + (a_first ? pb : pa);
  p.ds = (int)(a_first ? da : db);
  p.dl = (int)(a_first ? db : da);
  return p;
}

// first position in [lo, hi) of L with L[pos] >= x
__device__ __forceinline__ int lower_bound_i32(const int32_t* __restrict__ L, int lo, int hi, int32_t x) {
  while (lo < hi) {
    const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
    if (__ldg(L + mid) < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

struct HeurAcc {
  int cnt;
  double aa, ra;
};

// probes S[j] for j = j0, j0 + step, ... < j1 into L[lo, hi). S is sorted, so each probe starts where the last one ended.
__device__ __forceinline__ void probe(const int64_t* __restrict__ ptr, const int32_t* __restrict__ S, int j0, int j1, int step,
                                      const int32_t* __restrict__ L, int lo, int hi, HeurAcc& acc) {
  for (int j = j0; j < j1; j += step) {
    const int32_t x = __ldg(S + j);
    lo = lower_bound_i32(L, lo, hi, x);
    if (lo < hi && __ldg(L + lo) == x) {
      const int64_t d = __ldg(ptr + x + 1) - __ldg(ptr + x);   // >= 1: x is a neighbour
      acc.cnt += 1;
      acc.aa += d > 1 ? 1.0 / log((double)d) : 0.0;
      acc.ra += 1.0 / (double)d;
    }
  }
}

__device__ __forceinline__ bool id_ok(int64_t x, int64_t N) { return x >= 0 && x < N; }

// per pair: chunks[i] = ceil(w / CHUNK) when its probe count w = min(d(u), d(v)) exceeds LONG, else 0;
// info[0] += bad ids, info[2] += probes
__global__ void __launch_bounds__(kHeurThreads) k_lh_plan(const int64_t* __restrict__ ptr, int64_t N, const int64_t* __restrict__ u,
                                                          int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                          int64_t* __restrict__ chunks, unsigned long long* __restrict__ info) {
  int nbad = 0;
  unsigned long long probes = 0;
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i - lane < P; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < P) {
      const int64_t a = u[i * s_u], b = v[i * s_v];
      const bool oka = id_ok(a, N), okb = id_ok(b, N);
      nbad += !oka + !okb;
      int64_t w = 0;
      if (oka && okb) {
        const int64_t da = ptr[a + 1] - ptr[a], db = ptr[b + 1] - ptr[b];
        w = da < db ? da : db;
      }
      probes += (unsigned long long)w;
      chunks[i] = w > kHeurLong ? (w + kHeurChunk - 1) / kHeurChunk : 0;
    }
  }
  nbad = warp_sum_i(nbad);
#pragma unroll
  for (int o = 16; o; o >>= 1) probes += __shfl_xor_sync(0xffffffffu, probes, o);
  if (lane == 0 && nbad) atomicAdd(info + 0, (unsigned long long)nbad);
  if (lane == 0 && probes) atomicAdd(info + 2, probes);
}

// one warp per chunk: pair = the last i with chunk_off[i] <= c, chunk k = c - chunk_off[i] covers S[k CHUNK, (k+1) CHUNK)
__global__ void __launch_bounds__(kHeurThreads) k_lh_chunks(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                            const int64_t* __restrict__ u, int64_t s_u, const int64_t* __restrict__ v,
                                                            int64_t s_v, int64_t P, const int64_t* __restrict__ chunk_off,
                                                            int64_t n_chunks, int32_t* __restrict__ p_cnt, double* __restrict__ p_aa,
                                                            double* __restrict__ p_ra) {
  const int lane = threadIdx.x & 31;
  for (int64_t c = (int64_t)blockIdx.x * kHeurWarps + (threadIdx.x >> 5); c < n_chunks; c += (int64_t)gridDim.x * kHeurWarps) {
    int64_t lo = 0, hi = P - 1;   // chunk_off[0] = 0 <= c
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (chunk_off[mid] <= c)
        lo = mid;
      else
        hi = mid - 1;
    }
    const int64_t k = c - chunk_off[lo];
    int64_t da, db;
    const PairLists pl = pair_lists(ptr, adj, u[lo * s_u], v[lo * s_v], &da, &db);
    const int j0 = (int)(k * kHeurChunk);
    const int j1 = j0 + kHeurChunk < pl.ds ? j0 + kHeurChunk : pl.ds;
    // the chunk's range in the longer list: [first >= S[j0], first > S[j1 - 1])
    int bound = 0;
    if (lane == 0) bound = lower_bound_i32(pl.L, 0, pl.dl, __ldg(pl.S + j0));
    if (lane == 1) bound = lower_bound_i32(pl.L, 0, pl.dl, __ldg(pl.S + j1 - 1) + 1);   // ids < 2^31 - 1
    const int llo = __shfl_sync(0xffffffffu, bound, 0), lhi = __shfl_sync(0xffffffffu, bound, 1);
    HeurAcc acc{0, 0.0, 0.0};
    probe(ptr, pl.S, j0 + lane, j1, 32, pl.L, llo, lhi, acc);
    acc.cnt = warp_sum_i(acc.cnt);
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      acc.aa += __shfl_xor_sync(0xffffffffu, acc.aa, o);
      acc.ra += __shfl_xor_sync(0xffffffffu, acc.ra, o);
    }
    if (lane == 0) p_cnt[c] = acc.cnt, p_aa[c] = acc.aa, p_ra[c] = acc.ra;
  }
}

// one 8-lane group per pair: intersect a short pair, or add a chunked pair's partials in chunk order; write the four scores
__global__ void __launch_bounds__(kHeurThreads) k_lh_pairs(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t N,
                                                           const int64_t* __restrict__ u, int64_t s_u, const int64_t* __restrict__ v,
                                                           int64_t s_v, int64_t P, const int64_t* __restrict__ chunk_off,
                                                           const int32_t* __restrict__ p_cnt, const double* __restrict__ p_aa,
                                                           const double* __restrict__ p_ra, float* __restrict__ out) {
  const int g = (threadIdx.x & 31) / kHeurGroup, gl = threadIdx.x & (kHeurGroup - 1);
  const int64_t stride = (int64_t)gridDim.x * kHeurGroups;
  // the loop bound is warp-uniform so that every lane reaches the shuffles below
  for (int64_t base = (int64_t)blockIdx.x * kHeurGroups + (threadIdx.x >> 5) * (32 / kHeurGroup); base < P; base += stride) {
    const int64_t i = base + g;
    HeurAcc acc{0, 0.0, 0.0};
    bool valid = false;
    int64_t da = 0, db = 0;
    if (i < P) {
      const int64_t a = u[i * s_u], b = v[i * s_v];
      valid = id_ok(a, N) && id_ok(b, N);
      if (valid) {
        const PairLists pl = pair_lists(ptr, adj, a, b, &da, &db);
        if (pl.ds > kHeurLong) {
          if (gl == 0)
            for (int64_t c = chunk_off[i], e = chunk_off[i + 1]; c < e; ++c) acc.cnt += p_cnt[c], acc.aa += p_aa[c], acc.ra += p_ra[c];
        } else {
          probe(ptr, pl.S, gl, pl.ds, kHeurGroup, pl.L, 0, pl.dl, acc);
        }
      }
    }
#pragma unroll
    for (int o = kHeurGroup / 2; o; o >>= 1) {
      acc.cnt += __shfl_xor_sync(0xffffffffu, acc.cnt, o);
      acc.aa += __shfl_xor_sync(0xffffffffu, acc.aa, o);
      acc.ra += __shfl_xor_sync(0xffffffffu, acc.ra, o);
    }
    if (i < P && gl == 0) {
      float cn = __int_as_float(0x7fc00000), jac = cn, aa = cn, ra = cn;   // NaN for a pair with a bad id
      if (valid) {
        const int64_t den = da + db - acc.cnt;
        cn = (float)acc.cnt;
        jac = den > 0 ? __fdiv_rn(cn, (float)den) : 0.f;
        aa = __double2float_rn(acc.aa);
        ra = __double2float_rn(acc.ra);
      }
      out[i] = cn, out[P + i] = jac, out[2 * P + i] = aa, out[3 * P + i] = ra;
    }
  }
}

}  // namespace twowl

using namespace twowl;

extern "C" size_t twowl_simple_adjacency_workspace_bytes(int64_t n_edges) {
  const int64_t M = n_edges > 0 ? 2 * n_edges : 1;
  return 4 * align_up((size_t)M * sizeof(uint32_t)) + align_up(radix_workspace_bytes(M)) +
         align_up((size_t)(M + 1) * sizeof(int64_t)) + align_up(scan_workspace_bytes(M));
}

extern "C" int twowl_simple_adjacency(const int64_t* row, int64_t s_row, const int64_t* col, int64_t s_col, int64_t n_edges,
                                      int64_t num_nodes, int64_t* ptr, int32_t* adj, int32_t* bad, void* ws, size_t ws_bytes,
                                      void* stream) {
  TW_CHECK_ARG(n_edges >= 0 && n_edges < 0x40000000LL && num_nodes >= 0 && num_nodes < 0x7fffffffLL,
               "simple_adjacency: bad sizes (0 <= n_edges < 2^30, 0 <= num_nodes < 2^31 - 1)");
  TW_CHECK_ARG(ptr && bad && (n_edges == 0 || (row && col && adj)), "simple_adjacency: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_simple_adjacency_workspace_bytes(n_edges));
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(bad, 0, sizeof(int32_t), s));
  if (n_edges == 0) {
    TW_CUDA(cudaMemsetAsync(ptr, 0, (size_t)(num_nodes + 1) * sizeof(int64_t), s));
    return 0;
  }
  const int64_t M = 2 * n_edges;
  Carver c(ws);
  uint32_t* k0 = c.take<uint32_t>(M);
  uint32_t* v0 = c.take<uint32_t>(M);
  uint32_t* k1 = c.take<uint32_t>(M);
  uint32_t* v1 = c.take<uint32_t>(M);
  void* rws = c.take<char>(radix_workspace_bytes(M));
  int64_t* pos = c.take<int64_t>(M + 1);
  void* sws = c.take<char>(scan_workspace_bytes(M));
  const int bits = bits_for_value(num_nodes);   // rows run up to the sentinel N
  k_adj_keys<<<grid_for(n_edges, kHeurThreads), kHeurThreads, 0, s>>>(row, s_row, col, s_col, n_edges, num_nodes, k0, v0, bad);
  TW_LAUNCH_CHECK();
  // stable LSD order: by neighbour, then by row -> entries ordered by (row, neighbour)
  if (int rc = radix_sort_pairs(k0, v0, k1, v1, M, bits, rws, s)) return rc;    // k1 = neighbour (sorted), v1 = row
  if (int rc = radix_sort_pairs(v1, k1, k0, v0, M, bits, rws, s)) return rc;    // k0 = row (sorted), v0 = neighbour
  const uint32_t N32 = (uint32_t)num_nodes;
  const int grid = grid_for(M, kHeurThreads);
  k_adj_flags<<<grid, kHeurThreads, 0, s>>>(k0, v0, M, N32, pos);
  TW_LAUNCH_CHECK();
  if (int rc = scan_exclusive_i64(pos, pos, M, sws, s)) return rc;
  k_adj_fill<<<grid, kHeurThreads, 0, s>>>(k0, v0, M, N32, pos, adj);
  k_adj_ptr<<<grid_for(num_nodes + 1, kHeurThreads), kHeurThreads, 0, s>>>(k0, M, num_nodes, pos, ptr);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_link_plan_workspace_bytes(int64_t P) { return scan_workspace_bytes(P > 0 ? P : 1); }

extern "C" int twowl_link_plan(const int64_t* ptr, int64_t num_nodes, const int64_t* u, int64_t s_u, const int64_t* v, int64_t s_v,
                               int64_t P, int64_t* chunk_off, int64_t* info, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(P >= 0 && P < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL,
               "link_plan: bad sizes (0 <= P < 2^31, 0 <= num_nodes < 2^31 - 1)");
  TW_CHECK_ARG(ptr && chunk_off && info && (P == 0 || (u && v)), "link_plan: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_link_plan_workspace_bytes(P));
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(info, 0, 3 * sizeof(int64_t), s));
  if (P > 0) {
    k_lh_plan<<<grid_for(P, kHeurThreads), kHeurThreads, 0, s>>>(ptr, num_nodes, u, s_u, v, s_v, P, chunk_off,
                                                                 reinterpret_cast<unsigned long long*>(info));
    TW_LAUNCH_CHECK();
  }
  if (int rc = scan_exclusive_i64(chunk_off, chunk_off, P, ws, s)) return rc;
  TW_CUDA(cudaMemcpyAsync(info + 1, chunk_off + P, sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
  return 0;
}

extern "C" size_t twowl_link_heuristics_workspace_bytes(int64_t n_chunks) {
  const size_t m = (size_t)(n_chunks > 0 ? n_chunks : 1);
  return align_up(m * sizeof(int32_t)) + 2 * align_up(m * sizeof(double));
}

extern "C" int twowl_link_heuristics(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* u, int64_t s_u,
                                     const int64_t* v, int64_t s_v, int64_t P, const int64_t* chunk_off, int64_t n_chunks, float* out,
                                     void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(P >= 0 && P < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL && n_chunks >= 0,
               "link_heuristics: bad sizes (0 <= P < 2^31, 0 <= num_nodes < 2^31 - 1, n_chunks >= 0)");
  TW_CHECK_ARG(ptr && (P == 0 || (u && v && chunk_off && out)), "link_heuristics: null pointer");   // adj: NULL when nnz = 0
  TW_CHECK_WS(ws_bytes, twowl_link_heuristics_workspace_bytes(n_chunks));
  if (P == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t m = (size_t)(n_chunks > 0 ? n_chunks : 1);
  Carver c(ws);
  int32_t* p_cnt = c.take<int32_t>(m);
  double* p_aa = c.take<double>(m);
  double* p_ra = c.take<double>(m);
  if (n_chunks > 0) {
    k_lh_chunks<<<grid_for(n_chunks, kHeurWarps), kHeurThreads, 0, s>>>(ptr, adj, u, s_u, v, s_v, P, chunk_off, n_chunks, p_cnt, p_aa,
                                                                        p_ra);
    TW_LAUNCH_CHECK();
  }
  k_lh_pairs<<<grid_for(P, kHeurGroups), kHeurThreads, 0, s>>>(ptr, adj, num_nodes, u, s_u, v, s_v, P, chunk_off, p_cnt, p_aa, p_ra, out);
  TW_LAUNCH_CHECK();
  return 0;
}
