// sampler.cu - seeded uniform sampling of NON-EDGES without the dense N x N mask of the reference
// (TwoWL/utils.py:129-146 builds a [N, N] uint8 mask - 1 TB at 1 M nodes - and takes a random subset of its nonzeros;
// TwoWL/operators/datasets.py:176-197 calls PyG's negative_sampling, which draws from the same set with python's random.sample).
// Same output contract: `count` DISTINCT pairs, uniform over the pairs that are not in the given edge list (and are not self
// loops), in the upper triangle (row < col) for the undirected split or as ordered pairs for negative_sampling.
//
// One open-addressing hash set over the 64-bit keys row * N + col holds the edges and, as they are accepted, the samples:
//   insert   every edge with owner -1 (an edge always wins)
//   round r  every unresolved slot i draws its candidate from a counter-based generator keyed by (seed, i, r) and claims it with
//            atomicMin(owner, i); after the round a slot whose candidate is owned by itself is final (owner := -1), every other
//            slot draws again in round r + 1
// The winner of a key is the SMALLEST slot that proposed it - a function of (seed, edges) only, so the output is reproducible
// whatever the thread timing; only the cell a key lands in depends on the race, never who owns it. HBM-bound integer work.
//
// The same table and rounds draw per-source negatives for ranking evaluation (OGB's "filtered" tail corruption): slot j of row
// i = j / k draws a node w uniform over [0, N), drops it when w == src[i] or the undirected edge {src[i], w} is in the table, and
// otherwise claims the key N^2 + i N + w - past every edge key, so one table holds both - so that a row never holds w twice.
#include "common.cuh"

namespace twowl {

constexpr int kSmpThreads = 256;
constexpr long long kEmpty = -1;

__device__ __forceinline__ uint64_t smp_mix(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t smp_slot(uint64_t key, uint64_t mask) { return smp_mix(key + 0x9E3779B97F4A7C15ull) & mask; }

// claim `key` for `owner` (smaller owner wins); linear probing
__device__ __forceinline__ void smp_claim(long long* __restrict__ keys, int* __restrict__ owners, uint64_t mask, long long key, int owner) {
  uint64_t h = smp_slot((uint64_t)key, mask);
  for (;;) {
    const long long prev = atomicCAS(reinterpret_cast<unsigned long long*>(keys + h), (unsigned long long)kEmpty, (unsigned long long)key);
    if (prev == kEmpty || prev == key) {
      atomicMin(owners + h, owner);
      return;
    }
    h = (h + 1) & mask;
  }
}
__device__ __forceinline__ int* smp_find(const long long* __restrict__ keys, int* __restrict__ owners, uint64_t mask, long long key) {
  uint64_t h = smp_slot((uint64_t)key, mask);
  for (;;) {
    const long long k = keys[h];
    if (k == key) return owners + h;
    if (k == kEmpty) return nullptr;
    h = (h + 1) & mask;
  }
}

__global__ void __launch_bounds__(kSmpThreads) k_smp_insert_edges(const int64_t* __restrict__ row, int64_t s_row,
                                                                  const int64_t* __restrict__ col, int64_t s_col, int64_t n_edges,
                                                                  int64_t N, int undirected, long long* __restrict__ keys,
                                                                  int* __restrict__ owners, uint64_t mask) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = row[e * s_row], c = col[e * s_col];
    if (r < 0 || c < 0 || r >= N || c >= N) continue;
    if (undirected && r > c) {
      const int64_t t = r;
      r = c, c = t;
    }
    smp_claim(keys, owners, mask, (long long)(r * N + c), -1);
  }
}

// candidate of slot i in round r: an ordered pair uniform over [0,N)^2 (64-bit multiply-high range reduction); undirected: sorted
__device__ __forceinline__ long long smp_candidate(uint64_t seed, int64_t i, int round, int64_t N, int undirected) {
  const uint64_t a = smp_mix(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(2 * i + 1) + ((uint64_t)round << 40));
  const uint64_t b = smp_mix(a ^ 0xD1B54A32D192ED03ull);
  int64_t r = (int64_t)__umul64hi(a, (uint64_t)N), c = (int64_t)__umul64hi(b, (uint64_t)N);
  if (r == c) return -1;                       // self loop: never a sample (the callers pass the graph with its self loops added)
  if (undirected && r > c) {
    const int64_t t = r;
    r = c, c = t;
  }
  return (long long)(r * N + c);
}

__global__ void __launch_bounds__(kSmpThreads) k_smp_propose(uint64_t seed, int round, int64_t count, int64_t N, int undirected,
                                                             const uint8_t* __restrict__ done, long long* __restrict__ cand,
                                                             long long* __restrict__ keys, int* __restrict__ owners, uint64_t mask) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    if (done[i]) continue;
    const long long key = smp_candidate(seed, i, round, N, undirected);
    cand[i] = key;
    if (key >= 0) smp_claim(keys, owners, mask, key, (int)i);
  }
}

__global__ void __launch_bounds__(kSmpThreads) k_smp_resolve(int64_t count, int64_t N, uint8_t* __restrict__ done,
                                                             const long long* __restrict__ cand, const long long* __restrict__ keys,
                                                             int* __restrict__ owners, uint64_t mask, int64_t* __restrict__ out_row,
                                                             int64_t* __restrict__ out_col, int* __restrict__ unresolved) {
  int left = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    if (done[i]) continue;
    const long long key = cand[i];
    int* own = key >= 0 ? smp_find(keys, owners, mask, key) : nullptr;
    if (own && *own == (int)i) {
      *own = -1;                               // final: no later round may take this key
      done[i] = 1;
      if (out_row) out_row[i] = key / N;
      out_col[i] = key % N;
    } else {
      ++left;
    }
  }
  left = __reduce_add_sync(0xffffffffu, left);
  if ((threadIdx.x & 31) == 0 && left) atomicAdd(unresolved, left);
}

// slot j of row i = j / k: candidate w uniform over [0,N); key N^2 + i N + w unless w is src[i] or a neighbour of it (then -1)
__global__ void __launch_bounds__(kSmpThreads) k_tail_propose(uint64_t seed, int round, int64_t count, int64_t k, int64_t N,
                                                              const int64_t* __restrict__ src, const uint8_t* __restrict__ done,
                                                              long long* __restrict__ cand, long long* __restrict__ keys,
                                                              int* __restrict__ owners, uint64_t mask) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += (int64_t)gridDim.x * blockDim.x) {
    if (done[j]) continue;
    const int64_t i = j / k, u = src[i];
    const uint64_t a = smp_mix(seed + 0x9E3779B97F4A7C15ull * (uint64_t)(2 * j + 1) + ((uint64_t)round << 40));
    const int64_t w = (int64_t)__umul64hi(a, (uint64_t)N);
    long long key = -1;
    if (u >= 0 && u < N && w != u) {
      const long long edge = (long long)(u < w ? u * N + w : w * N + u);
      // every key below N^2 in the table is an edge, inserted by an earlier kernel; the concurrent claims only fill empty cells
      if (!smp_find(keys, owners, mask, edge)) key = (long long)(N * N + i * N + w);
    }
    cand[j] = key;
    if (key >= 0) smp_claim(keys, owners, mask, key, (int)j);
  }
}

static uint64_t smp_capacity(int64_t n_edges, int64_t count) {
  uint64_t need = 2ull * (uint64_t)(n_edges + count) + 1024ull, cap = 1024;
  while (cap < need) cap <<= 1;
  return cap;
}

}  // namespace twowl

using namespace twowl;

extern "C" size_t twowl_nonedge_sample_workspace_bytes(int64_t n_edges, int64_t count) {
  const uint64_t cap = smp_capacity(n_edges > 0 ? n_edges : 0, count > 0 ? count : 0);
  const size_t c = (size_t)(count > 0 ? count : 1);
  return align_up(cap * sizeof(long long)) + align_up(cap * sizeof(int)) + align_up(c * sizeof(long long)) + align_up(c);
}

extern "C" int twowl_nonedge_sample(const int64_t* row, int64_t s_row, const int64_t* col, int64_t s_col, int64_t n_edges,
                                    int64_t num_nodes, int64_t count, int32_t undirected, uint64_t seed, int32_t rounds,
                                    int64_t* out_row, int64_t* out_col, uint8_t* done_out, int32_t* unresolved, void* ws,
                                    size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(n_edges >= 0 && count >= 0 && num_nodes > 0 && rounds > 0, "nonedge_sample: bad sizes");
  TW_CHECK_ARG(count < 0x7fffffffLL && num_nodes < (1LL << 31), "nonedge_sample: count and num_nodes must be below 2^31");
  TW_CHECK_ARG(unresolved != nullptr && (count == 0 || (out_row && out_col)), "nonedge_sample: null output");
  TW_CHECK_WS(ws_bytes, twowl_nonedge_sample_workspace_bytes(n_edges, count));
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(unresolved, 0, sizeof(int32_t), s));
  if (count == 0) return 0;
  const uint64_t cap = smp_capacity(n_edges, count), mask = cap - 1;
  Carver c(ws);
  long long* keys = c.take<long long>(cap);
  int* owners = c.take<int>(cap);
  long long* cand = c.take<long long>((size_t)count);
  uint8_t* done = c.take<uint8_t>((size_t)count);
  TW_CUDA(cudaMemsetAsync(keys, 0xFF, cap * sizeof(long long), s));
  TW_CUDA(cudaMemsetAsync(owners, 0x7F, cap * sizeof(int), s));
  TW_CUDA(cudaMemsetAsync(done, 0, (size_t)count, s));
  if (n_edges > 0) {
    k_smp_insert_edges<<<grid_for(n_edges, kSmpThreads), kSmpThreads, 0, s>>>(row, s_row, col, s_col, n_edges, num_nodes, undirected, keys,
                                                                            owners, mask);
    TW_LAUNCH_CHECK();
  }
  for (int r = 0; r < rounds; ++r) {
    TW_CUDA(cudaMemsetAsync(unresolved, 0, sizeof(int32_t), s));
    k_smp_propose<<<grid_for(count, kSmpThreads), kSmpThreads, 0, s>>>(seed, r, count, num_nodes, undirected, done, cand, keys, owners, mask);
    k_smp_resolve<<<grid_for(count, kSmpThreads), kSmpThreads, 0, s>>>(count, num_nodes, done, cand, keys, owners, mask, out_row, out_col,
                                                                       unresolved);
    TW_LAUNCH_CHECK();
  }
  if (done_out) TW_CUDA(cudaMemcpyAsync(done_out, done, (size_t)count, cudaMemcpyDeviceToDevice, s));
  return 0;
}

extern "C" size_t twowl_tail_negative_sample_workspace_bytes(int64_t n_edges, int64_t P, int64_t k) {
  const int64_t count = (P > 0 && k > 0) ? P * k : 0;
  return twowl_nonedge_sample_workspace_bytes(n_edges, count);
}

extern "C" int twowl_tail_negative_sample(const int64_t* row, int64_t s_row, const int64_t* col, int64_t s_col, int64_t n_edges,
                                          int64_t num_nodes, const int64_t* src, int64_t P, int64_t k, uint64_t seed, int32_t rounds,
                                          int64_t* out, int32_t* unresolved, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(n_edges >= 0 && P >= 0 && k >= 1 && num_nodes > 0 && rounds > 0, "tail_negative_sample: bad sizes");
  TW_CHECK_ARG(P < 0x7fffffffLL && k < 0x7fffffffLL && P * k < 0x7fffffffLL && num_nodes < (1LL << 31),
               "tail_negative_sample: P * k and num_nodes must be below 2^31");
  TW_CHECK_ARG(unresolved != nullptr && (P == 0 || (src && out)) && (n_edges == 0 || (row && col)),
               "tail_negative_sample: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_tail_negative_sample_workspace_bytes(n_edges, P, k));
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(unresolved, 0, sizeof(int32_t), s));
  const int64_t count = P * k;
  if (count == 0) return 0;
  const uint64_t cap = smp_capacity(n_edges, count), mask = cap - 1;
  Carver c(ws);
  long long* keys = c.take<long long>(cap);
  int* owners = c.take<int>(cap);
  long long* cand = c.take<long long>((size_t)count);
  uint8_t* done = c.take<uint8_t>((size_t)count);
  TW_CUDA(cudaMemsetAsync(keys, 0xFF, cap * sizeof(long long), s));
  TW_CUDA(cudaMemsetAsync(owners, 0x7F, cap * sizeof(int), s));
  TW_CUDA(cudaMemsetAsync(done, 0, (size_t)count, s));
  TW_CUDA(cudaMemsetAsync(out, 0xFF, (size_t)count * sizeof(int64_t), s));     // -1 = unfilled
  if (n_edges > 0) {
    k_smp_insert_edges<<<grid_for(n_edges, kSmpThreads), kSmpThreads, 0, s>>>(row, s_row, col, s_col, n_edges, num_nodes, 1, keys,
                                                                            owners, mask);
    TW_LAUNCH_CHECK();
  }
  for (int r = 0; r < rounds; ++r) {
    TW_CUDA(cudaMemsetAsync(unresolved, 0, sizeof(int32_t), s));
    k_tail_propose<<<grid_for(count, kSmpThreads), kSmpThreads, 0, s>>>(seed, r, count, k, num_nodes, src, done, cand, keys, owners, mask);
    k_smp_resolve<<<grid_for(count, kSmpThreads), kSmpThreads, 0, s>>>(count, num_nodes, done, cand, keys, owners, mask, nullptr, out,
                                                                       unresolved);
    TW_LAUNCH_CHECK();
  }
  return 0;
}
