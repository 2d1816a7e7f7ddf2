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

// adds the terms of one common neighbour of degree d >= 1: Adamic-Adar 1 / ln d (0 for d = 1) and resource allocation 1 / d.
// The pair scores (probe) and the recommendations (k_rec_runs) both add them here, so the two ops see the same term bits.
__device__ __forceinline__ void heur_add(int64_t d, HeurAcc& acc) {
  acc.cnt += 1;
  acc.aa += d > 1 ? 1.0 / log((double)d) : 0.0;
  acc.ra += 1.0 / (double)d;
}

// probes S[j] for j = j0, j0 + step, ... < j1 into L[lo, hi). S is sorted, so each probe starts where the last one ended.
__device__ __forceinline__ void probe(const int64_t* __restrict__ ptr, const int32_t* __restrict__ S, int j0, int j1, int step,
                                      const int32_t* __restrict__ L, int lo, int hi, HeurAcc& acc) {
  for (int j = j0; j < j1; j += step) {
    const int32_t x = __ldg(S + j);
    lo = lower_bound_i32(L, lo, hi, x);
    if (lo < hi && __ldg(L + lo) == x) heur_add(__ldg(ptr + x + 1) - __ldg(ptr + x), acc);   // d >= 1: x is a neighbour
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

// ---------------------------------------------------------------- link recommendation ---------------
// The candidates of a source s are its two-hop non-neighbours. One batch of queries [q_begin, q_end), with M expansion entries:
//   expand   for j in the batch, w in N(s_j) ascending, v in N(w) ascending: entry e = (v, w), at the query's offset. The
//            batch's neighbour lists are cut into tiles of kRecTile; a CTA takes a tile, scans its degrees and writes the
//            tile's entries flat, so a hub's row and a hub neighbour's long list both spread over the whole CTA.
//   sort     stably by v, then stably by the query: entries ordered by (query, v, e), so each (query, v) run lists its
//            common neighbours w in ascending order.
//   runs     the head of a run drops v = s and v in N(s) (binary search), else sums its w terms in order, one thread per
//            run, and keys the run by its chosen score (descending: the complement of the fp32 bits, every score > 0).
//   top-k    stably by that key, then stably by the query: each query's runs in (score descending, v ascending) order.
//            Query j's rows are the first k entries of its segment, found by binary search.
// Every position is a uint32, so a batch holds fewer than 2^31 entries. No floating-point atomics; the order of every sum is
// fixed by the sorts, which are stable: the result is bitwise repeatable and does not depend on how queries are batched.
constexpr int kRecThreads = 256;
constexpr int kRecTile = kRecThreads;                  // neighbours of a source per expansion tile
constexpr uint32_t kRecDead = 0xffffffffu;             // score key of an entry that is not a kept run head

__device__ __forceinline__ int64_t deg_of(const int64_t* __restrict__ ptr, int64_t x) { return __ldg(ptr + x + 1) - __ldg(ptr + x); }

// largest i in [0, n) with off[i] - base <= x, given off[0] - base <= x
__device__ __forceinline__ int64_t last_le(const int64_t* __restrict__ off, int64_t n, int64_t base, int64_t x) {
  int64_t lo = 0, hi = n - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (off[mid] - base <= x)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

// first position in [0, n) of the ascending keys with keys[pos] >= x
__device__ __forceinline__ int64_t lower_bound_u32(const uint32_t* __restrict__ keys, int64_t n, uint32_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

__device__ __forceinline__ int64_t warp_sum_l(int64_t v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// exclusive scan of one value per thread over the CTA; *total = the CTA's sum. sm: kRecThreads / 32 + 1 slots.
__device__ __forceinline__ int64_t block_exclusive_scan_l(int64_t v, int64_t* total, int64_t* sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int64_t o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) sm[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int64_t w = lane < kRecThreads / 32 ? sm[lane] : 0;
    int64_t winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int64_t o = __shfl_up_sync(0xffffffffu, winc, d);
      if (lane >= d) winc += o;
    }
    if (lane < kRecThreads / 32) sm[lane] = winc - w;
    if (lane == kRecThreads / 32 - 1) sm[kRecThreads / 32] = winc;
  }
  __syncthreads();
  const int64_t res = sm[warp] + inc - v;
  *total = sm[kRecThreads / 32];
  __syncthreads();
  return res;
}

// one warp per query: xcount[q] = X(s) = sum of d(w) over w in N(s), 0 for a bad id; info[0] += bad ids
__global__ void __launch_bounds__(kRecThreads) k_rec_plan(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t N,
                                                          const int64_t* __restrict__ src, int64_t s_src, int64_t Q,
                                                          int64_t* __restrict__ xcount, unsigned long long* __restrict__ info) {
  const int lane = threadIdx.x & 31;
  for (int64_t q = (int64_t)blockIdx.x * (kRecThreads / 32) + (threadIdx.x >> 5); q < Q; q += (int64_t)gridDim.x * (kRecThreads / 32)) {
    const int64_t s = src[q * s_src];
    const bool ok = id_ok(s, N);
    int64_t x = 0;
    if (ok)
      for (int64_t i = ptr[s] + lane, e = ptr[s + 1]; i < e; i += 32) x += deg_of(ptr, __ldg(adj + i));
    x = warp_sum_l(x);
    if (lane == 0) {
      xcount[q] = x;
      if (!ok) atomicAdd(info, 1ull);
    }
  }
}

// tile_cnt[j] = ceil(d(s_j) / kRecTile) for the batch's queries
__global__ void __launch_bounds__(kRecThreads) k_rec_tiles(const int64_t* __restrict__ ptr, const int64_t* __restrict__ src, int64_t s_src,
                                                           int64_t Qb, int64_t* __restrict__ tile_cnt) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < Qb; j += (int64_t)gridDim.x * blockDim.x)
    tile_cnt[j] = (deg_of(ptr, src[j * s_src]) + kRecTile - 1) / kRecTile;
}

struct RecTile {
  int64_t s, first;   // the source, and the position in N(s) of the tile's first neighbour
  int n;              // neighbours in the tile
};

// tile `it` < tile_off[Qb]: query = the last j with tile_off[j] <= it
__device__ __forceinline__ RecTile rec_tile(const int64_t* __restrict__ ptr, const int64_t* __restrict__ src, int64_t s_src, int64_t Qb,
                                            const int64_t* __restrict__ tile_off, int64_t it) {
  const int64_t j = last_le(tile_off, Qb, 0, it);
  RecTile t;
  t.s = src[j * s_src];
  t.first = (it - tile_off[j]) * kRecTile;
  const int64_t rest = deg_of(ptr, t.s) - t.first;
  t.n = (int)(rest < kRecTile ? rest : kRecTile);
  return t;
}

// one CTA per tile: tile_sum[it] = the number of entries the tile expands to (0 for it >= the batch's tile count)
__global__ void __launch_bounds__(kRecThreads) k_rec_tile_sums(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                               const int64_t* __restrict__ src, int64_t s_src, int64_t Qb,
                                                               const int64_t* __restrict__ tile_off, int64_t n_items,
                                                               int64_t* __restrict__ tile_sum) {
  __shared__ int64_t sm[kRecThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n_tiles = tile_off[Qb];
  for (int64_t it = blockIdx.x; it < n_items; it += gridDim.x) {
    int64_t x = 0;
    if (it < n_tiles) {
      const RecTile t = rec_tile(ptr, src, s_src, Qb, tile_off, it);
      if ((int)threadIdx.x < t.n) x = deg_of(ptr, __ldg(adj + ptr[t.s] + t.first + threadIdx.x));
    }
    x = warp_sum_l(x);
    if (lane == 0) sm[warp] = x;
    __syncthreads();
    if (threadIdx.x == 0) {
      int64_t tot = 0;
#pragma unroll
      for (int w = 0; w < kRecThreads / 32; ++w) tot += sm[w];
      tile_sum[it] = tot;
    }
    __syncthreads();
  }
}

// one CTA per tile: entry base + x of the tile = (v, w) with w the tile's neighbour whose list covers x; key = v, val = entry
__global__ void __launch_bounds__(kRecThreads) k_rec_expand(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                            const int64_t* __restrict__ src, int64_t s_src, int64_t Qb,
                                                            const int64_t* __restrict__ tile_off, const int64_t* __restrict__ tile_base,
                                                            uint32_t* __restrict__ key, uint32_t* __restrict__ val,
                                                            uint32_t* __restrict__ V, uint32_t* __restrict__ W) {
  __shared__ int64_t off[kRecThreads], nb[kRecThreads], sm[kRecThreads / 32 + 1];
  __shared__ int32_t wid[kRecThreads];
  const int64_t n_tiles = tile_off[Qb];
  for (int64_t it = blockIdx.x; it < n_tiles; it += gridDim.x) {
    const RecTile t = rec_tile(ptr, src, s_src, Qb, tile_off, it);
    int64_t dw = 0;
    if ((int)threadIdx.x < t.n) {
      const int32_t w = __ldg(adj + ptr[t.s] + t.first + threadIdx.x);
      wid[threadIdx.x] = w;
      nb[threadIdx.x] = ptr[w];
      dw = ptr[w + 1] - nb[threadIdx.x];
    }
    int64_t total;
    off[threadIdx.x] = block_exclusive_scan_l(dw, &total, sm);   // ends in a barrier: off / wid / nb are visible
    __syncthreads();
    const int64_t base = tile_base[it];
    for (int64_t x = threadIdx.x; x < total; x += kRecThreads) {
      int lo = 0, hi = kRecThreads - 1;                           // the last neighbour whose offset is <= x (it has d > 0)
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= x)
          lo = mid;
        else
          hi = mid - 1;
      }
      const uint32_t v = (uint32_t)__ldg(adj + nb[lo] + (x - off[lo]));
      const int64_t e = base + x;
      key[e] = v, V[e] = v, W[e] = (uint32_t)wid[lo], val[e] = (uint32_t)e;
    }
    __syncthreads();
  }
}

// after the sort by v (val = entry): key = the entry's batch-local query (the last j with exp_off[j] - exp_off[0] <= entry)
__global__ void __launch_bounds__(kRecThreads) k_rec_qkeys(const uint32_t* __restrict__ ent, int64_t M, const int64_t* __restrict__ exp_off,
                                                           int64_t Qb, uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  const int64_t base = exp_off[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t e = ent[i];
    key[i] = (uint32_t)last_le(exp_off, Qb, base, e);
    val[i] = e;
  }
}

// entries in (query, v, e) order: qk = query, ent = entry. A kept run head r gets the run's scores sc[r] and the key of the
// chosen score; every other position the key kRecDead. key / val feed the sort by score (val = position).
__global__ void __launch_bounds__(kRecThreads) k_rec_runs(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                          const int64_t* __restrict__ src, int64_t s_src, const uint32_t* __restrict__ qk,
                                                          const uint32_t* __restrict__ ent, const uint32_t* __restrict__ V,
                                                          const uint32_t* __restrict__ W, int64_t M, int by, float4* __restrict__ sc,
                                                          uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t j = qk[r], v = V[ent[r]];
    uint32_t k = kRecDead;
    if (r == 0 || qk[r - 1] != j || V[ent[r - 1]] != v) {
      const int64_t s = src[(int64_t)j * s_src];
      const int64_t ps = ptr[s], ds = ptr[s + 1] - ps;
      const int lo = lower_bound_i32(adj + ps, 0, (int)ds, (int32_t)v);
      if ((int64_t)v != s && !(lo < ds && __ldg(adj + ps + lo) == (int32_t)v)) {
        HeurAcc acc{0, 0.0, 0.0};
        for (int64_t q = r; q < M && qk[q] == j && V[ent[q]] == v; ++q) heur_add(deg_of(ptr, W[ent[q]]), acc);   // w ascending
        const int64_t den = ds + deg_of(ptr, v) - acc.cnt;
        const float cn = (float)acc.cnt;
        const float4 o = make_float4(cn, den > 0 ? __fdiv_rn(cn, (float)den) : 0.f, __double2float_rn(acc.aa),
                                     __double2float_rn(acc.ra));
        sc[r] = o;
        k = ~__float_as_uint(by == 0 ? o.x : by == 1 ? o.y : by == 2 ? o.z : o.w);
      }
    }
    key[r] = k;
    val[r] = (uint32_t)r;
  }
}

// after the sort by score key (skey, pos): key = the query of a kept run, Qb (last) for the rest; val = position
__global__ void __launch_bounds__(kRecThreads) k_rec_jkeys(const uint32_t* __restrict__ skey, const uint32_t* __restrict__ pos,
                                                           const uint32_t* __restrict__ qk, int64_t M, uint32_t Qb,
                                                           uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t p = pos[i];
    key[i] = skey[i] != kRecDead ? qk[p] : Qb;
    val[i] = p;
  }
}

// one thread per output slot (j, t): the t-th run of query j's segment in the final order, or padding (-1, NaN)
__global__ void __launch_bounds__(kRecThreads) k_rec_out(const uint32_t* __restrict__ fkey, const uint32_t* __restrict__ fpos, int64_t M,
                                                         const uint32_t* __restrict__ ent, const uint32_t* __restrict__ V,
                                                         const float4* __restrict__ sc, int64_t Qb, int64_t k, int64_t q_begin, int64_t QK,
                                                         int64_t* __restrict__ ids, float* __restrict__ scores) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < Qb * k; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / k, t = i - j * k;
    const int64_t lo = lower_bound_u32(fkey, M, (uint32_t)j), hi = lower_bound_u32(fkey, M, (uint32_t)j + 1);
    const int64_t o = q_begin * k + i;
    if (lo + t < hi) {
      const uint32_t r = fpos[lo + t];
      const float4 s = sc[r];
      ids[o] = V[ent[r]];
      scores[o] = s.x, scores[QK + o] = s.y, scores[2 * QK + o] = s.z, scores[3 * QK + o] = s.w;
    } else {
      const float nan = __int_as_float(0x7fc00000);
      ids[o] = -1;
      scores[o] = nan, scores[QK + o] = nan, scores[2 * QK + o] = nan, scores[3 * QK + o] = nan;
    }
  }
}

// ---------------------------------------------------------------- common-neighbour lists -------------
// The same decomposition as link_heuristics (twowl_link_plan's chunk_off): a short pair is probed by one 8-lane group, a long
// pair's chunks by one warp each. An entry mask (uint8 per adjacency entry, NULL = none) deletes entries: a probe from a masked
// entry of the shorter list finds nothing, and a hit on a masked entry of the longer list does not count.
//   count  chunk counts into chunk_base[c], then pair counts (a long pair adds its chunks) into cn_ptr[i]; both scanned.
//   fill   a round probes one strided position per lane; a group ballot ranks the hits, so they are written in probe order,
//          which is ascending id order. A long pair's chunk c writes from cn_ptr[i] + chunk_base[c] - chunk_base[chunk_off[i]].

// probes S[j] into L[lo, hi) (lo advances: S is sorted); true when S[j] is a common neighbour that no mask deletes
__device__ __forceinline__ bool cn_probe(const int32_t* __restrict__ S, const uint8_t* __restrict__ mS, int j, const int32_t* __restrict__ L,
                                         const uint8_t* __restrict__ mL, int& lo, int hi) {
  if (mS && __ldg(mS + j)) return false;
  const int32_t x = __ldg(S + j);
  lo = lower_bound_i32(L, lo, hi, x);
  return lo < hi && __ldg(L + lo) == x && !(mL && __ldg(mL + lo));
}

// the mask pointers of a pair's two lists (NULL without a mask)
__device__ __forceinline__ void cn_masks(const int32_t* __restrict__ adj, const uint8_t* __restrict__ mask, const PairLists& pl,
                                         const uint8_t** mS, const uint8_t** mL) {
  *mS = mask ? mask + (pl.S - adj) : nullptr;
  *mL = mask ? mask + (pl.L - adj) : nullptr;
}

struct CnChunk {
  int64_t pair;
  PairLists pl;
  int j0, j1, llo, lhi;
};

// one warp per chunk c: its pair, probe range and the matching range of the longer list (k_lh_chunks' merge path)
__device__ __forceinline__ CnChunk cn_chunk(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, const int64_t* __restrict__ u,
                                            int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                            const int64_t* __restrict__ chunk_off, int64_t c) {
  const int lane = threadIdx.x & 31;
  CnChunk ch;
  ch.pair = last_le(chunk_off, P, 0, c);
  const int64_t k = c - chunk_off[ch.pair];
  int64_t da, db;
  ch.pl = pair_lists(ptr, adj, u[ch.pair * s_u], v[ch.pair * s_v], &da, &db);
  ch.j0 = (int)(k * kHeurChunk);
  ch.j1 = ch.j0 + kHeurChunk < ch.pl.ds ? ch.j0 + kHeurChunk : ch.pl.ds;
  int bound = 0;
  if (lane == 0) bound = lower_bound_i32(ch.pl.L, 0, ch.pl.dl, __ldg(ch.pl.S + ch.j0));
  if (lane == 1) bound = lower_bound_i32(ch.pl.L, 0, ch.pl.dl, __ldg(ch.pl.S + ch.j1 - 1) + 1);   // ids < 2^31 - 1
  ch.llo = __shfl_sync(0xffffffffu, bound, 0);
  ch.lhi = __shfl_sync(0xffffffffu, bound, 1);
  return ch;
}

__global__ void __launch_bounds__(kHeurThreads) k_cn_chunk_count(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                                 const uint8_t* __restrict__ mask, const int64_t* __restrict__ u,
                                                                 int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                                 const int64_t* __restrict__ chunk_off, int64_t n_chunks,
                                                                 int64_t* __restrict__ chunk_cnt) {
  const int lane = threadIdx.x & 31;
  for (int64_t c = (int64_t)blockIdx.x * kHeurWarps + (threadIdx.x >> 5); c < n_chunks; c += (int64_t)gridDim.x * kHeurWarps) {
    const CnChunk ch = cn_chunk(ptr, adj, u, s_u, v, s_v, P, chunk_off, c);
    const uint8_t *mS, *mL;
    cn_masks(adj, mask, ch.pl, &mS, &mL);
    int cnt = 0, lo = ch.llo;
    for (int j = ch.j0 + lane; j < ch.j1; j += 32) cnt += cn_probe(ch.pl.S, mS, j, ch.pl.L, mL, lo, ch.lhi);
    cnt = warp_sum_i(cnt);
    if (lane == 0) chunk_cnt[c] = cnt;
  }
}

// one 8-lane group per pair: the count of a short pair, or the sum of a long pair's chunk counts (0 for a bad id)
__global__ void __launch_bounds__(kHeurThreads) k_cn_pair_count(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                                const uint8_t* __restrict__ mask, int64_t N, const int64_t* __restrict__ u,
                                                                int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                                const int64_t* __restrict__ chunk_off, const int64_t* __restrict__ chunk_cnt,
                                                                int64_t* __restrict__ cnt_out) {
  const int g = (threadIdx.x & 31) / kHeurGroup, gl = threadIdx.x & (kHeurGroup - 1);
  const int64_t stride = (int64_t)gridDim.x * kHeurGroups;
  // the loop bound is warp-uniform so that every lane reaches the shuffles below
  for (int64_t base = (int64_t)blockIdx.x * kHeurGroups + (threadIdx.x >> 5) * (32 / kHeurGroup); base < P; base += stride) {
    const int64_t i = base + g;
    int64_t cnt = 0;
    if (i < P) {
      const int64_t a = u[i * s_u], b = v[i * s_v];
      if (id_ok(a, N) && id_ok(b, N)) {
        int64_t da, db;
        const PairLists pl = pair_lists(ptr, adj, a, b, &da, &db);
        if (pl.ds > kHeurLong) {
          if (gl == 0)
            for (int64_t c = chunk_off[i], e = chunk_off[i + 1]; c < e; ++c) cnt += chunk_cnt[c];
        } else {
          const uint8_t *mS, *mL;
          cn_masks(adj, mask, pl, &mS, &mL);
          int lo = 0;
          for (int j = gl; j < pl.ds; j += kHeurGroup) cnt += cn_probe(pl.S, mS, j, pl.L, mL, lo, pl.dl);
        }
      }
    }
#pragma unroll
    for (int o = kHeurGroup / 2; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (i < P && gl == 0) cnt_out[i] = cnt;
  }
}

// one warp per chunk of a long pair: its common neighbours from the chunk's base, in ascending order
__global__ void __launch_bounds__(kHeurThreads) k_cn_chunk_fill(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                                const uint8_t* __restrict__ mask, const int64_t* __restrict__ u,
                                                                int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                                const int64_t* __restrict__ chunk_off, int64_t n_chunks,
                                                                const int64_t* __restrict__ cn_ptr, const int64_t* __restrict__ chunk_base,
                                                                int32_t* __restrict__ ids, int32_t* __restrict__ pair) {
  const int lane = threadIdx.x & 31;
  const unsigned below = (1u << lane) - 1u;
  for (int64_t c = (int64_t)blockIdx.x * kHeurWarps + (threadIdx.x >> 5); c < n_chunks; c += (int64_t)gridDim.x * kHeurWarps) {
    const CnChunk ch = cn_chunk(ptr, adj, u, s_u, v, s_v, P, chunk_off, c);
    const uint8_t *mS, *mL;
    cn_masks(adj, mask, ch.pl, &mS, &mL);
    int64_t out = cn_ptr[ch.pair] + chunk_base[c] - chunk_base[chunk_off[ch.pair]];
    int lo = ch.llo;
    for (int j0 = ch.j0; j0 < ch.j1; j0 += 32) {   // warp-uniform rounds
      const int j = j0 + lane;
      const bool hit = j < ch.j1 && cn_probe(ch.pl.S, mS, j, ch.pl.L, mL, lo, ch.lhi);
      const unsigned b = __ballot_sync(0xffffffffu, hit);
      if (hit) {
        const int64_t e = out + __popc(b & below);
        ids[e] = __ldg(ch.pl.S + j);
        pair[e] = (int32_t)ch.pair;
      }
      out += __popc(b);
    }
  }
}

// one 8-lane group per short pair: its common neighbours from cn_ptr[i], in ascending order (long pairs: k_cn_chunk_fill)
__global__ void __launch_bounds__(kHeurThreads) k_cn_pair_fill(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj,
                                                               const uint8_t* __restrict__ mask, int64_t N, const int64_t* __restrict__ u,
                                                               int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                               const int64_t* __restrict__ cn_ptr, int32_t* __restrict__ ids,
                                                               int32_t* __restrict__ pair) {
  const int lane = threadIdx.x & 31, g = lane / kHeurGroup, gl = lane & (kHeurGroup - 1);
  const unsigned gmask = 0xffu << (g * kHeurGroup), below = (1u << lane) - 1u;
  for (int64_t i = ((int64_t)blockIdx.x * kHeurThreads + threadIdx.x) / kHeurGroup; i < P; i += (int64_t)gridDim.x * kHeurGroups) {
    const int64_t a = u[i * s_u], b = v[i * s_v];
    if (!id_ok(a, N) || !id_ok(b, N)) continue;                 // uniform over the group, as is every branch below
    int64_t da, db;
    const PairLists pl = pair_lists(ptr, adj, a, b, &da, &db);
    if (pl.ds > kHeurLong) continue;
    const uint8_t *mS, *mL;
    cn_masks(adj, mask, pl, &mS, &mL);
    int64_t out = cn_ptr[i];
    int lo = 0;
    for (int j0 = 0; j0 < pl.ds; j0 += kHeurGroup) {            // group-uniform rounds
      const int j = j0 + gl;
      const bool hit = j < pl.ds && cn_probe(pl.S, mS, j, pl.L, mL, lo, pl.dl);
      const unsigned bal = __ballot_sync(gmask, hit) & gmask;
      if (hit) {
        const int64_t e = out + __popc(bal & below);
        ids[e] = __ldg(pl.S + j);
        pair[e] = (int32_t)i;
      }
      out += __popc(bal);
    }
  }
}

// one thread per pair (u, v), u != v, both valid: mask the entry of v in N(u) and the entry of u in N(v), each where it exists
// (on the symmetric simple adjacency: both, exactly when the pair is an edge); info[0] += bad ids
__global__ void __launch_bounds__(kHeurThreads) k_adj_pair_mask(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t N,
                                                                const int64_t* __restrict__ u, int64_t s_u, const int64_t* __restrict__ v,
                                                                int64_t s_v, int64_t P, uint8_t* __restrict__ mask,
                                                                unsigned long long* __restrict__ info) {
  int nbad = 0;
  const int lane = threadIdx.x & 31;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i - lane < P; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < P) {
      const int64_t a = u[i * s_u], b = v[i * s_v];
      const bool oka = id_ok(a, N), okb = id_ok(b, N);
      nbad += !oka + !okb;
      if (oka && okb && a != b) {
        const int64_t pa = ptr[a], pb = ptr[b];
        const int da = (int)(ptr[a + 1] - pa), db = (int)(ptr[b + 1] - pb);
        // each direction is looked up and checked on its own, so that a CSR that is not symmetric marks only entries it holds
        const int ia = lower_bound_i32(adj + pa, 0, da, (int32_t)b);
        if (ia < da && __ldg(adj + pa + ia) == (int32_t)b) mask[pa + ia] = 1;
        const int ib = lower_bound_i32(adj + pb, 0, db, (int32_t)a);
        if (ib < db && __ldg(adj + pb + ib) == (int32_t)a) mask[pb + ib] = 1;
      }
    }
  }
  nbad = warp_sum_i(nbad);
  if (lane == 0 && nbad) atomicAdd(info, (unsigned long long)nbad);
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

extern "C" size_t twowl_recommend_plan_workspace_bytes(int64_t Q) { return scan_workspace_bytes(Q > 0 ? Q : 1); }

extern "C" int twowl_recommend_plan(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* src, int64_t s_src, int64_t Q,
                                    int64_t* exp_off, int64_t* info, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(Q >= 0 && Q < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL,
               "recommend_plan: bad sizes (0 <= Q < 2^31, 0 <= num_nodes < 2^31 - 1)");
  TW_CHECK_ARG(ptr && exp_off && info && (Q == 0 || src), "recommend_plan: null pointer");   // adj: NULL when nnz = 0
  TW_CHECK_WS(ws_bytes, twowl_recommend_plan_workspace_bytes(Q));
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(info, 0, 2 * sizeof(int64_t), s));
  if (Q > 0) {
    k_rec_plan<<<grid_for(Q, kRecThreads / 32), kRecThreads, 0, s>>>(ptr, adj, num_nodes, src, s_src, Q, exp_off,
                                                                     reinterpret_cast<unsigned long long*>(info));
    TW_LAUNCH_CHECK();
  }
  if (int rc = scan_exclusive_i64(exp_off, exp_off, Q, ws, s)) return rc;
  TW_CUDA(cudaMemcpyAsync(info + 1, exp_off + Q, sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
  return 0;
}

// expansion tiles of a batch: at most one partial tile per query plus M / kRecTile full ones (each neighbour w has d(w) >= 1)
static int64_t rec_items(int64_t M, int64_t Qb) { return Qb + cdiv(M, kRecTile); }

extern "C" size_t twowl_recommend_workspace_bytes(int64_t n_entries, int64_t n_queries) {
  const int64_t M = n_entries > 0 ? n_entries : 1, Qb = n_queries > 0 ? n_queries : 1, T = rec_items(M, Qb);
  return 7 * align_up((size_t)M * sizeof(uint32_t)) + align_up((size_t)M * sizeof(float4)) + align_up(radix_workspace_bytes(M)) +
         align_up((size_t)(Qb + 1) * sizeof(int64_t)) + align_up(scan_workspace_bytes(Qb)) + align_up((size_t)(T + 1) * sizeof(int64_t)) +
         align_up(scan_workspace_bytes(T));
}

extern "C" int twowl_recommend(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* src, int64_t s_src, int64_t Q,
                               int64_t q_begin, int64_t q_end, const int64_t* exp_off, int64_t n_entries, int32_t by, int64_t k,
                               int64_t* ids, float* scores, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(Q >= 0 && Q < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL && 0 <= q_begin && q_begin <= q_end && q_end <= Q,
               "recommend: bad sizes (0 <= q_begin <= q_end <= Q < 2^31, 0 <= num_nodes < 2^31 - 1)");
  TW_CHECK_ARG(k >= 1 && k < 0x7fffffffLL && Q * k < (1LL << 60), "recommend: k must be in [1, 2^31) with Q * k < 2^60");
  TW_CHECK_ARG(by >= 0 && by < 4, "recommend: by must be 0 (cn), 1 (jaccard), 2 (aa) or 3 (ra)");
  TW_CHECK_ARG(n_entries >= 0 && n_entries < 0x80000000LL, "recommend: a batch must expand to 0 <= n_entries < 2^31 entries");
  TW_CHECK_ARG(ptr && exp_off && ids && scores && (q_begin == q_end || src) && (n_entries == 0 || adj), "recommend: null pointer");
  const int64_t Qb = q_end - q_begin, M = n_entries;
  TW_CHECK_WS(ws_bytes, twowl_recommend_workspace_bytes(M, Qb));
  if (Qb == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t* bsrc = src + q_begin * s_src;
  const int64_t* boff = exp_off + q_begin;
  Carver c(ws);
  uint32_t* A = c.take<uint32_t>(M);
  uint32_t* B = c.take<uint32_t>(M);
  uint32_t* C = c.take<uint32_t>(M);
  uint32_t* D = c.take<uint32_t>(M);
  uint32_t* V = c.take<uint32_t>(M);
  uint32_t* W = c.take<uint32_t>(M);
  uint32_t* F = c.take<uint32_t>(M);
  float4* SC = c.take<float4>(M);
  void* rws = c.take<char>(radix_workspace_bytes(M));
  int64_t* tile_off = c.take<int64_t>(Qb + 1);
  void* tws = c.take<char>(scan_workspace_bytes(Qb));
  const int64_t T = rec_items(M, Qb);
  int64_t* tile_base = c.take<int64_t>(T + 1);
  void* bws = c.take<char>(scan_workspace_bytes(T));
  if (M > 0) {
    k_rec_tiles<<<grid_for(Qb, kRecThreads), kRecThreads, 0, s>>>(ptr, bsrc, s_src, Qb, tile_off);
    TW_LAUNCH_CHECK();
    if (int rc = scan_exclusive_i64(tile_off, tile_off, Qb, tws, s)) return rc;
    k_rec_tile_sums<<<grid_for(T, 1), kRecThreads, 0, s>>>(ptr, adj, bsrc, s_src, Qb, tile_off, T, tile_base);
    TW_LAUNCH_CHECK();
    if (int rc = scan_exclusive_i64(tile_base, tile_base, T, bws, s)) return rc;
    k_rec_expand<<<grid_for(T, 1), kRecThreads, 0, s>>>(ptr, adj, bsrc, s_src, Qb, tile_off, tile_base, A, B, V, W);
    TW_LAUNCH_CHECK();
    const int grid = grid_for(M, kRecThreads);
    // (query, v, entry) order: stably by v, then stably by the query
    if (int rc = radix_sort_pairs(A, B, C, D, M, bits_for_value(num_nodes - 1), rws, s)) return rc;   // C = v, D = entry
    k_rec_qkeys<<<grid, kRecThreads, 0, s>>>(D, M, boff, Qb, A, B);
    TW_LAUNCH_CHECK();
    if (int rc = radix_sort_pairs(A, B, C, D, M, bits_for_value(Qb - 1), rws, s)) return rc;          // C = query, D = entry
    k_rec_runs<<<grid, kRecThreads, 0, s>>>(ptr, adj, bsrc, s_src, C, D, V, W, M, by, SC, A, B);
    TW_LAUNCH_CHECK();
    // (query, score descending, v) order: stably by the score key, then stably by the query (the rest last)
    if (int rc = radix_sort_pairs(A, B, W, F, M, 32, rws, s)) return rc;                                // W = score key, F = position
    k_rec_jkeys<<<grid, kRecThreads, 0, s>>>(W, F, C, M, (uint32_t)Qb, A, B);
    TW_LAUNCH_CHECK();
    if (int rc = radix_sort_pairs(A, B, W, F, M, bits_for_value(Qb), rws, s)) return rc;              // W = query, F = position
  }
  k_rec_out<<<grid_for(Qb * k, kRecThreads), kRecThreads, 0, s>>>(W, F, M, D, V, SC, Qb, k, q_begin, Q * k, ids, scores);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_common_neighbors_count_workspace_bytes(int64_t P, int64_t n_chunks) {
  return align_up(scan_workspace_bytes(P > 0 ? P : 1)) + align_up(scan_workspace_bytes(n_chunks > 0 ? n_chunks : 1));
}

extern "C" int twowl_common_neighbors_count(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const uint8_t* entry_mask,
                                            const int64_t* u, int64_t s_u, const int64_t* v, int64_t s_v, int64_t P,
                                            const int64_t* chunk_off, int64_t n_chunks, int64_t* cn_ptr, int64_t* chunk_base, void* ws,
                                            size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(P >= 0 && P < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL && n_chunks >= 0,
               "common_neighbors_count: bad sizes (0 <= P < 2^31, 0 <= num_nodes < 2^31 - 1, n_chunks >= 0)");
  TW_CHECK_ARG(ptr && cn_ptr && chunk_base && (P == 0 || (u && v && chunk_off)), "common_neighbors_count: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_common_neighbors_count_workspace_bytes(P, n_chunks));
  cudaStream_t s = (cudaStream_t)stream;
  Carver c(ws);
  void* pws = c.take<char>(scan_workspace_bytes(P > 0 ? P : 1));
  void* cws = c.take<char>(scan_workspace_bytes(n_chunks > 0 ? n_chunks : 1));
  if (n_chunks > 0) {
    k_cn_chunk_count<<<grid_for(n_chunks, kHeurWarps), kHeurThreads, 0, s>>>(ptr, adj, entry_mask, u, s_u, v, s_v, P, chunk_off, n_chunks,
                                                                             chunk_base);
    TW_LAUNCH_CHECK();
  }
  if (P > 0) {
    k_cn_pair_count<<<grid_for(P, kHeurGroups), kHeurThreads, 0, s>>>(ptr, adj, entry_mask, num_nodes, u, s_u, v, s_v, P, chunk_off,
                                                                       chunk_base, cn_ptr);
    TW_LAUNCH_CHECK();
  }
  if (int rc = scan_exclusive_i64(cn_ptr, cn_ptr, P, pws, s)) return rc;
  if (int rc = scan_exclusive_i64(chunk_base, chunk_base, n_chunks, cws, s)) return rc;
  return 0;
}

extern "C" int twowl_common_neighbors_fill(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const uint8_t* entry_mask,
                                           const int64_t* u, int64_t s_u, const int64_t* v, int64_t s_v, int64_t P, const int64_t* chunk_off,
                                           int64_t n_chunks, const int64_t* cn_ptr, const int64_t* chunk_base, int64_t nnz_cn,
                                           int32_t* cn_ids, int32_t* cn_pair, void* stream) {
  TW_CHECK_ARG(P >= 0 && P < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL && n_chunks >= 0 && nnz_cn >= 0 &&
                   nnz_cn < 0x80000000LL,
               "common_neighbors_fill: bad sizes (0 <= P < 2^31, 0 <= num_nodes < 2^31 - 1, n_chunks >= 0, 0 <= nnz_cn < 2^31)");
  TW_CHECK_ARG(ptr && cn_ptr && chunk_base && (P == 0 || (u && v && chunk_off)) && (nnz_cn == 0 || (adj && cn_ids && cn_pair)),
               "common_neighbors_fill: null pointer");
  if (nnz_cn == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (n_chunks > 0) {
    k_cn_chunk_fill<<<grid_for(n_chunks, kHeurWarps), kHeurThreads, 0, s>>>(ptr, adj, entry_mask, u, s_u, v, s_v, P, chunk_off, n_chunks,
                                                                            cn_ptr, chunk_base, cn_ids, cn_pair);
    TW_LAUNCH_CHECK();
  }
  k_cn_pair_fill<<<grid_for(P, kHeurGroups), kHeurThreads, 0, s>>>(ptr, adj, entry_mask, num_nodes, u, s_u, v, s_v, P, cn_ptr, cn_ids,
                                                                    cn_pair);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_adjacency_pair_mask(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, int64_t nnz, const int64_t* u,
                                         int64_t s_u, const int64_t* v, int64_t s_v, int64_t P, uint8_t* mask, int64_t* info,
                                         void* stream) {
  TW_CHECK_ARG(P >= 0 && P < 0x7fffffffLL && num_nodes >= 0 && num_nodes < 0x7fffffffLL && nnz >= 0,
               "adjacency_pair_mask: bad sizes (0 <= P < 2^31, 0 <= num_nodes < 2^31 - 1, nnz >= 0)");
  TW_CHECK_ARG(ptr && info && (P == 0 || (u && v)) && (nnz == 0 || (adj && mask)), "adjacency_pair_mask: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(info, 0, sizeof(int64_t), s));
  if (nnz > 0) TW_CUDA(cudaMemsetAsync(mask, 0, (size_t)nnz, s));
  if (P > 0) {
    k_adj_pair_mask<<<grid_for(P, kHeurThreads), kHeurThreads, 0, s>>>(ptr, adj, num_nodes, u, s_u, v, s_v, P, mask,
                                                                       reinterpret_cast<unsigned long long*>(info));
    TW_LAUNCH_CHECK();
  }
  return 0;
}
