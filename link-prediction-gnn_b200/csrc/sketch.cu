// sketch.cu - BUDDY's subgraph sketches (Chamberlain et al., ICLR 2023): per-node MinHash and HyperLogLog rows of the d-hop
// neighbourhoods, built by segmented min / max over a simple adjacency, and the per-pair distance-count features read from them.
// See include/twowl.h (twowl_sketch_*) for the definitions.
//
// A node's sketch row is V = num_perm / 4 + m / 16 16-byte vectors: the MinHash row (combined by an elementwise min of uint32) and
// the HyperLogLog row (a bytewise max). A hop is one gather over the adjacency. A 16-lane group takes one row, slice after slice,
// a slice being 16 consecutive vectors (256 bytes), and streams the slice of every neighbour with four loads in flight per lane.
// Rows longer than `chunk` entries are listed by a plan kernel and cut into chunks: each (chunk, slice) item writes a partial
// row into the workspace and a second pass combines a row's partials with its own row. min and max are exact, so the result does
// not depend on the cut.
#include "common.cuh"

namespace twowl {

namespace {

constexpr int kSkThreads = 256;
constexpr int kSkGroup = 16;                          // lanes per (row, slice) item
constexpr int kSkGroups = kSkThreads / kSkGroup;
constexpr int kSkFeatWarps = 4;                       // pairs per CTA of the feature kernel

struct SkHop {
  const int64_t* ptr;
  const int32_t* adj;
  const uint8_t* mask;
  int64_t N;
  int64_t chunk;
  int num_perm, m, vm, V, S;                          // vm = MinHash vectors per row, V = all vectors, S = slices per row
  const uint8_t* mh_in;
  const uint8_t* hll_in;
  uint8_t* mh_out;
  uint8_t* hll_out;
  const int32_t* counts;                              // [2]: long rows, chunks
  const int32_t* long_row;
  const int32_t* long_base;
  const int32_t* chunk_owner;
  uint4* partial;                                     // [chunk_cap, V]
  int64_t long_cap, chunk_cap;
};

// the lane's vector k of a row: where it lives (byte offset in the row of mh or hll), and how it combines
struct SkLane {
  bool on, is_min;
  const uint8_t* in;                                  // base of vector k in row 0 of the input
  uint8_t* out;
  int64_t stride;                                     // bytes per row
  uint4 ident;
};

__device__ __forceinline__ SkLane sk_lane(const SkHop& a, int k) {
  SkLane l;
  l.on = k < a.V;
  l.is_min = k < a.vm;
  if (l.is_min) {
    l.in = a.mh_in + (int64_t)k * 16;
    l.out = a.mh_out + (int64_t)k * 16;
    l.stride = (int64_t)a.num_perm * 4;
    l.ident = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
  } else {
    l.in = a.hll_in + (int64_t)(k - a.vm) * 16;
    l.out = a.hll_out + (int64_t)(k - a.vm) * 16;
    l.stride = a.m;
    l.ident = make_uint4(0u, 0u, 0u, 0u);
  }
  return l;
}

__device__ __forceinline__ uint4 sk_comb(const uint4& x, const uint4& y, bool is_min) {
  if (is_min) return make_uint4(min(x.x, y.x), min(x.y, y.y), min(x.z, y.z), min(x.w, y.w));
  return make_uint4(__vmaxu4(x.x, y.x), __vmaxu4(x.y, y.y), __vmaxu4(x.z, y.z), __vmaxu4(x.w, y.w));
}

__device__ __forceinline__ uint4 sk_load(const SkLane& l, int64_t row) {
  return __ldg(reinterpret_cast<const uint4*>(l.in + row * l.stride));
}

// acc combined with the lane's vector of every unmasked neighbour in entries [kb, ke). The group reads 16 ids at a time, one per
// lane, and hands them round by shuffles; every lane of the group runs the same loop (bounds are group-uniform).
__device__ __forceinline__ uint4 sk_gather(const SkHop& a, const SkLane& l, int64_t kb, int64_t ke, uint4 acc, unsigned gmask, int gl) {
  for (int64_t k0 = kb; k0 < ke; k0 += kSkGroup) {
    const int64_t k = k0 + gl;
    int w = -1;
    if (k < ke && !(a.mask && __ldg(a.mask + k))) w = __ldg(a.adj + k);
    const int cnt = ke - k0 < kSkGroup ? (int)(ke - k0) : kSkGroup;
    for (int j = 0; j < cnt; j += 4) {
      uint4 x[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int wt = __shfl_sync(gmask, w, j + t, kSkGroup);
        x[t] = (l.on && wt >= 0) ? sk_load(l, wt) : l.ident;
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) acc = sk_comb(acc, x[t], l.is_min);
    }
  }
  return acc;
}

__device__ __forceinline__ void sk_store(const SkLane& l, int64_t row, const uint4& v) {
  *reinterpret_cast<uint4*>(l.out + row * l.stride) = v;
}

// one row of at most `chunk` entries per group, slice after slice: own row combined with every neighbour's, written out
__global__ void __launch_bounds__(kSkThreads) k_sketch_rows(SkHop a) {
  const int gl = threadIdx.x & (kSkGroup - 1);
  const unsigned gmask = 0xffffu << (threadIdx.x & 16);
  for (int64_t r = ((int64_t)blockIdx.x * kSkThreads + threadIdx.x) / kSkGroup; r < a.N; r += (int64_t)gridDim.x * kSkGroups) {
    const int64_t kb = a.ptr[r], ke = a.ptr[r + 1];
    if (ke - kb > a.chunk) continue;                  // a long row: k_sketch_chunks + k_sketch_long
    for (int s = 0; s < a.S; ++s) {
      const SkLane l = sk_lane(a, s * kSkGroup + gl);
      uint4 acc = l.on ? sk_load(l, r) : l.ident;
      acc = sk_gather(a, l, kb, ke, acc, gmask, gl);
      if (l.on) sk_store(l, r, acc);
    }
  }
}

// one (chunk, slice) item per group: the chunk's neighbours combined into partial[chunk]
__global__ void __launch_bounds__(kSkThreads) k_sketch_chunks(SkHop a) {
  const int gl = threadIdx.x & (kSkGroup - 1);
  const unsigned gmask = 0xffffu << (threadIdx.x & 16);
  const int64_t items = (int64_t)a.counts[1] * a.S;
  for (int64_t it = ((int64_t)blockIdx.x * kSkThreads + threadIdx.x) / kSkGroup; it < items; it += (int64_t)gridDim.x * kSkGroups) {
    const int64_t c = it / a.S;
    const int s = (int)(it - c * a.S);
    const int slot = a.chunk_owner[c];
    const int64_t r = a.long_row[slot];
    const int64_t kb = a.ptr[r] + (c - a.long_base[slot]) * a.chunk;
    const int64_t ke = kb + a.chunk < a.ptr[r + 1] ? kb + a.chunk : a.ptr[r + 1];
    const int k = s * kSkGroup + gl;
    const SkLane l = sk_lane(a, k);
    const uint4 acc = sk_gather(a, l, kb, ke, l.ident, gmask, gl);
    if (l.on) a.partial[c * a.V + k] = acc;
  }
}

// one (long row, slice) item per group: own row combined with the row's chunk partials, in chunk order
__global__ void __launch_bounds__(kSkThreads) k_sketch_long(SkHop a) {
  const int gl = threadIdx.x & (kSkGroup - 1);
  const int64_t items = (int64_t)a.counts[0] * a.S;
  for (int64_t it = ((int64_t)blockIdx.x * kSkThreads + threadIdx.x) / kSkGroup; it < items; it += (int64_t)gridDim.x * kSkGroups) {
    const int64_t slot = it / a.S;
    const int s = (int)(it - slot * a.S);
    const int k = s * kSkGroup + gl;
    const SkLane l = sk_lane(a, k);
    if (!l.on) continue;
    const int64_t r = a.long_row[slot];
    const int64_t nch = (a.ptr[r + 1] - a.ptr[r] + a.chunk - 1) / a.chunk;
    uint4 acc = sk_load(l, r);
    for (int64_t c = a.long_base[slot], e = c + nch; c < e; ++c) acc = sk_comb(acc, a.partial[c * a.V + k], l.is_min);
    sk_store(l, r, acc);
  }
}

// rows longer than `chunk` entries, listed in any order (results never depend on it) with their first chunk
__global__ void __launch_bounds__(kSkThreads) k_sketch_plan(const int64_t* __restrict__ ptr, int64_t N, int64_t chunk,
                                                           int32_t* __restrict__ counts, int32_t* __restrict__ long_row,
                                                           int32_t* __restrict__ long_base, int32_t* __restrict__ chunk_owner) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t len = ptr[r + 1] - ptr[r];
    if (len > chunk) {
      const int nch = (int)((len + chunk - 1) / chunk);
      const int slot = atomicAdd(&counts[0], 1);
      const int base = atomicAdd(&counts[1], nch);
      long_row[slot] = (int32_t)r;
      long_base[slot] = base;
      for (int c = 0; c < nch; ++c) chunk_owner[base + c] = slot;
    }
  }
}

// hop 0: MinHash and HyperLogLog rows of {u}
__global__ void __launch_bounds__(kSkThreads) k_sketch_init(int64_t N, int num_perm, int p, uint64_t seed_mh, uint64_t seed_hll,
                                                           uint32_t* __restrict__ mh, uint4* __restrict__ hll) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = i0; i < N * num_perm; i += stride) {
    const int64_t u = i / num_perm, j = i - u * num_perm;
    mh[i] = hash_u32(seed_mh, ((uint64_t)j << 32) | (uint64_t)u);
  }
  const int vh = (1 << p) / 16;
  for (int64_t i = i0; i < N * vh; i += stride) {
    const int64_t u = i / vh;
    const int q = (int)(i - u * vh);
    const uint32_t h = hash_u32(seed_hll, (uint64_t)u);
    const uint32_t reg = h & ((1u << p) - 1u), w = h >> p;
    const uint32_t rank = w ? (uint32_t)(__clz(w) - p + 1) : (uint32_t)(33 - p);
    const uint32_t word = (int)(reg >> 4) == q ? (reg >> 2) & 3 : 4u, val = rank << (8 * (reg & 3));
    hll[i] = make_uint4(word == 0 ? val : 0u, word == 1 ? val : 0u, word == 2 ? val : 0u, word == 3 ? val : 0u);
  }
}

// ---------------------------------------------------------------- pair features -------------------------------------------

// the HyperLogLog estimate of the register row max(a, b) (b = NULL: a), on every lane of the warp. Z is a sum of dyadic terms
// >= 2^-33 over at most 1024 registers: 43 significant bits, exact in double in any order.
__device__ __forceinline__ double sk_est(const uint8_t* a, const uint8_t* b, int m, int p) {
  const int lane = threadIdx.x & 31;
  const uint32_t* a4 = reinterpret_cast<const uint32_t*>(a);
  const uint32_t* b4 = reinterpret_cast<const uint32_t*>(b);
  double z = 0.0;
  int zeros = 0;
  for (int j = lane; j < m / 4; j += 32) {
    uint32_t w = a4[j];
    if (b) w = __vmaxu4(w, b4[j]);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int r = (w >> (8 * t)) & 0xff;
      z += __longlong_as_double((long long)(1023 - r) << 52);   // 2^-r
      zeros += r == 0;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    z += __shfl_xor_sync(0xffffffffu, z, o);
    zeros += __shfl_xor_sync(0xffffffffu, zeros, o);
  }
  const double md = (double)m;
  const double alpha = m == 16 ? 0.673 : m == 32 ? 0.697 : m == 64 ? 0.709 : 0.7213 / (1.0 + 1.079 / md);
  if (zeros > 0) {
    const double thr = p == 4 ? 10.0 : p == 5 ? 20.0 : p == 6 ? 40.0 : p == 7 ? 80.0 : p == 8 ? 220.0 : p == 9 ? 400.0 : 900.0;
    const double lc = md * log(md / (double)zeros);
    if (lc <= thr) return lc;
  }
  return alpha * md * md / z;
}

// the fraction of equal entries of two MinHash rows (num_perm a multiple of 32), on every lane
__device__ __forceinline__ double sk_jaccard(const uint32_t* a, const uint32_t* b, int num_perm) {
  const int lane = threadIdx.x & 31;
  int eq = 0;
  for (int j = lane; j < num_perm; j += 32) eq += __popc(__ballot_sync(0xffffffffu, a[j] == b[j]));
  return (double)eq / (double)num_perm;
}

// one warp per pair. The warp's shared slice holds, per endpoint, the HyperLogLog rows of hops 0..k and the MinHash rows of hops
// 1..k, each read once from global memory; the k^2 (d1, d2) combinations are then formed from shared memory.
__global__ void __launch_bounds__(kSkFeatWarps * 32) k_sketch_features(int k, int64_t N, int num_perm, int p, const uint32_t* __restrict__ mh,
                                                                      const uint8_t* __restrict__ hll, const int64_t* __restrict__ u,
                                                                      int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                                      float* __restrict__ out, unsigned long long* __restrict__ info) {
  extern __shared__ uint4 sk_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int m = 1 << p;
  const int hll_bytes = (k + 1) * m, mh_bytes = k * num_perm * 4;
  const int side = hll_bytes + mh_bytes;
  uint8_t* base = reinterpret_cast<uint8_t*>(sk_smem) + (size_t)wib * 2 * side;
  const int nf = k * k + 2 * k;
  for (int64_t i = (int64_t)blockIdx.x * kSkFeatWarps + wib; i < P; i += (int64_t)gridDim.x * kSkFeatWarps) {
    const int64_t a = u[i * s_u], b = v[i * s_v];
    if (!(a >= 0 && a < N && b >= 0 && b < N)) {
      if (lane < nf) out[i * nf + lane] = 0.f;
      if (lane == 0) atomicAdd(info, 1ull);
      continue;
    }
    __syncwarp();                                     // the previous pair's reads of the slice are done
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int64_t x = e ? b : a;
      uint4* dst = reinterpret_cast<uint4*>(base + e * side);
      for (int d = 0; d <= k; ++d) {
        const uint4* src = reinterpret_cast<const uint4*>(hll + ((int64_t)d * N + x) * m);
        for (int q = lane; q < m / 16; q += 32) dst[d * (m / 16) + q] = __ldg(src + q);
      }
      uint4* dmh = reinterpret_cast<uint4*>(base + e * side + hll_bytes);
      for (int d = 1; d <= k; ++d) {
        const uint4* src = reinterpret_cast<const uint4*>(mh + ((int64_t)d * N + x) * num_perm);
        for (int q = lane; q < num_perm / 4; q += 32) dmh[(d - 1) * (num_perm / 4) + q] = __ldg(src + q);
      }
    }
    __syncwarp();
    const uint8_t* hu = base;
    const uint8_t* hv = base + side;
    const uint32_t* mu = reinterpret_cast<const uint32_t*>(base + hll_bytes);
    const uint32_t* mv = reinterpret_cast<const uint32_t*>(base + side + hll_bytes);
    double eu[TWOWL_SKETCH_MAX_HOPS + 1], ev[TWOWL_SKETCH_MAX_HOPS + 1];
    double I[TWOWL_SKETCH_MAX_HOPS + 1][TWOWL_SKETCH_MAX_HOPS + 1];
#pragma unroll
    for (int d = 0; d <= TWOWL_SKETCH_MAX_HOPS; ++d) {
      eu[d] = d <= k ? sk_est(hu + d * m, nullptr, m, p) : 0.0;
      ev[d] = d <= k ? sk_est(hv + d * m, nullptr, m, p) : 0.0;
      I[0][d] = I[d][0] = 0.0;
    }
#pragma unroll
    for (int d1 = 1; d1 <= TWOWL_SKETCH_MAX_HOPS; ++d1)
#pragma unroll
      for (int d2 = 1; d2 <= TWOWL_SKETCH_MAX_HOPS; ++d2)
        I[d1][d2] = (d1 <= k && d2 <= k) ? sk_jaccard(mu + (d1 - 1) * num_perm, mv + (d2 - 1) * num_perm, num_perm) *
                                               sk_est(hu + d1 * m, hv + d2 * m, m, p)
                                         : 0.0;
    double A[TWOWL_SKETCH_MAX_HOPS + 1][TWOWL_SKETCH_MAX_HOPS + 1];   // summed so that (v, u) gives the transpose bit for bit
#pragma unroll
    for (int d1 = 1; d1 <= TWOWL_SKETCH_MAX_HOPS; ++d1)
#pragma unroll
      for (int d2 = 1; d2 <= TWOWL_SKETCH_MAX_HOPS; ++d2) A[d1][d2] = (I[d1][d2] + I[d1 - 1][d2 - 1]) - (I[d1 - 1][d2] + I[d1][d2 - 1]);
    double val = 0.0;
#pragma unroll
    for (int d1 = 1; d1 <= TWOWL_SKETCH_MAX_HOPS; ++d1) {
      double su = 0.0, sv = 0.0;
#pragma unroll
      for (int d2 = 1; d2 <= TWOWL_SKETCH_MAX_HOPS; ++d2) {
        if (d2 <= k) {
          su += A[d1][d2];
          sv += A[d2][d1];
          if (d1 <= k && lane == (d1 - 1) * k + d2 - 1) val = A[d1][d2];
        }
      }
      if (d1 <= k && lane == k * k + d1 - 1) val = (eu[d1] - eu[d1 - 1]) - su;
      if (d1 <= k && lane == k * k + k + d1 - 1) val = (ev[d1] - ev[d1 - 1]) - sv;
    }
    if (lane < nf) out[i * nf + lane] = __double2float_rn(val > 0.0 ? val : 0.0);
  }
}

size_t sk_feat_smem(int k, int num_perm, int p) { return (size_t)kSkFeatWarps * 2 * ((size_t)(k + 1) * (1 << p) + (size_t)k * num_perm * 4); }

bool sk_params_ok(int32_t num_perm, int32_t hll_p) {
  return num_perm >= 32 && num_perm <= 1024 && num_perm % 32 == 0 && hll_p >= 4 && hll_p <= 10;
}

int64_t sk_long_cap(int64_t nnz, int64_t chunk) { return nnz / chunk + 1; }
int64_t sk_chunk_cap(int64_t nnz, int64_t chunk) { return 2 * (nnz / chunk) + 2; }

}  // namespace

}  // namespace twowl

using namespace twowl;

#define SK_CHECK_PARAMS(fn, num_perm, hll_p)                                                                                   \
  TW_CHECK_ARG(sk_params_ok(num_perm, hll_p), fn ": num_perm = %d must be a multiple of 32 in [32, 1024] and hll_p = %d in [4, 10]", \
               (int)(num_perm), (int)(hll_p))

extern "C" int twowl_sketch_init(int64_t num_nodes, int32_t num_perm, int32_t hll_p, uint64_t seed, int32_t* minhash, uint8_t* hll,
                                 void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL, "sketch_init: bad sizes (0 <= num_nodes < 2^31 - 1)");
  SK_CHECK_PARAMS("sketch_init", num_perm, hll_p);
  TW_CHECK_ARG(num_nodes == 0 || (minhash && hll), "sketch_init: null pointer");
  TW_CHECK_ARG(aligned16(minhash) && aligned16(hll), "sketch_init: sketch pointers must be 16-byte aligned");
  if (num_nodes == 0) return 0;
  const int64_t work = num_nodes * (num_perm > (1 << hll_p) / 16 ? num_perm : (1 << hll_p) / 16);
  k_sketch_init<<<grid_for(work, kSkThreads), kSkThreads, 0, (cudaStream_t)stream>>>(
      num_nodes, num_perm, hll_p, seed * 2, seed * 2 + 1, reinterpret_cast<uint32_t*>(minhash), reinterpret_cast<uint4*>(hll));
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_sketch_hop_workspace_bytes(int64_t nnz, int32_t num_perm, int32_t hll_p, int64_t chunk) {
  if (nnz < 0 || chunk < 1 || !sk_params_ok(num_perm, hll_p)) return 0;
  const int64_t lc = sk_long_cap(nnz, chunk), cc = sk_chunk_cap(nnz, chunk);
  const int64_t V = num_perm / 4 + (1 << hll_p) / 16;
  return align_up(2 * sizeof(int32_t)) + 2 * align_up(lc * sizeof(int32_t)) + align_up(cc * sizeof(int32_t)) +
         align_up((size_t)cc * V * sizeof(uint4));
}

extern "C" int twowl_sketch_hop(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, int64_t nnz, const uint8_t* entry_mask,
                                int32_t num_perm, int32_t hll_p, int64_t chunk, const int32_t* mh_in, const uint8_t* hll_in,
                                int32_t* mh_out, uint8_t* hll_out, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && nnz >= 0 && nnz < 0x80000000LL,
               "sketch_hop: bad sizes (0 <= num_nodes < 2^31 - 1, 0 <= nnz < 2^31)");
  SK_CHECK_PARAMS("sketch_hop", num_perm, hll_p);
  TW_CHECK_ARG(chunk >= 1 && chunk <= (1LL << 30), "sketch_hop: chunk = %lld outside [1, 2^30]", (long long)chunk);
  TW_CHECK_ARG(ptr && (nnz == 0 || adj) && (num_nodes == 0 || (mh_in && hll_in && mh_out && hll_out)), "sketch_hop: null pointer");
  TW_CHECK_ARG(aligned16(mh_in) && aligned16(hll_in) && aligned16(mh_out) && aligned16(hll_out),
               "sketch_hop: sketch pointers must be 16-byte aligned");
  TW_CHECK_ARG(num_nodes == 0 || ((const void*)mh_in != (const void*)mh_out && (const void*)hll_in != (const void*)hll_out),
               "sketch_hop: in and out must be different rows");
  TW_CHECK_WS(ws_bytes, twowl_sketch_hop_workspace_bytes(nnz, num_perm, hll_p, chunk));
  TW_CHECK_ARG(ws, "sketch_hop: null pointer");
  if (num_nodes == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  SkHop a;
  a.ptr = ptr;
  a.adj = adj;
  a.mask = entry_mask;
  a.N = num_nodes;
  a.chunk = chunk;
  a.num_perm = num_perm;
  a.m = 1 << hll_p;
  a.vm = num_perm / 4;
  a.V = a.vm + a.m / 16;
  a.S = (a.V + kSkGroup - 1) / kSkGroup;
  a.mh_in = reinterpret_cast<const uint8_t*>(mh_in);
  a.hll_in = hll_in;
  a.mh_out = reinterpret_cast<uint8_t*>(mh_out);
  a.hll_out = hll_out;
  a.long_cap = sk_long_cap(nnz, chunk);
  a.chunk_cap = sk_chunk_cap(nnz, chunk);
  Carver c(ws);
  int32_t* counts = c.take<int32_t>(2);
  int32_t* long_row = c.take<int32_t>(a.long_cap);
  int32_t* long_base = c.take<int32_t>(a.long_cap);
  int32_t* chunk_owner = c.take<int32_t>(a.chunk_cap);
  a.partial = c.take<uint4>((size_t)a.chunk_cap * a.V);
  a.counts = counts;
  a.long_row = long_row;
  a.long_base = long_base;
  a.chunk_owner = chunk_owner;
  TW_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), s));
  k_sketch_plan<<<grid_for(num_nodes, kSkThreads), kSkThreads, 0, s>>>(ptr, num_nodes, chunk, counts, long_row, long_base, chunk_owner);
  TW_LAUNCH_CHECK();
  k_sketch_chunks<<<grid_for(a.chunk_cap * a.S, kSkGroups), kSkThreads, 0, s>>>(a);
  TW_LAUNCH_CHECK();
  k_sketch_rows<<<grid_for(num_nodes, kSkGroups), kSkThreads, 0, s>>>(a);
  TW_LAUNCH_CHECK();
  k_sketch_long<<<grid_for(a.long_cap * a.S, kSkGroups), kSkThreads, 0, s>>>(a);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_sketch_pair_features(int32_t hops, int64_t num_nodes, int32_t num_perm, int32_t hll_p, const int32_t* minhash,
                                          const uint8_t* hll, const int64_t* u, int64_t s_u, const int64_t* v, int64_t s_v, int64_t P,
                                          float* out, int64_t* info, void* stream) {
  TW_CHECK_ARG(hops >= 1 && hops <= TWOWL_SKETCH_MAX_HOPS, "sketch_pair_features: hops = %d outside [1, %d]", (int)hops,
               TWOWL_SKETCH_MAX_HOPS);
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && P >= 0 && P < 0x80000000LL,
               "sketch_pair_features: bad sizes (0 <= num_nodes < 2^31 - 1, 0 <= P < 2^31)");
  SK_CHECK_PARAMS("sketch_pair_features", num_perm, hll_p);
  TW_CHECK_ARG(info && (P == 0 || (u && v && out)) && (num_nodes == 0 || (minhash && hll)), "sketch_pair_features: null pointer");
  TW_CHECK_ARG(aligned16(minhash) && aligned16(hll), "sketch_pair_features: sketch pointers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(info, 0, sizeof(int64_t), s));
  if (P == 0) return 0;
  const size_t smem = sk_feat_smem(hops, num_perm, hll_p);
  if (smem > 48 * 1024) TW_CUDA(cudaFuncSetAttribute(k_sketch_features, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_sketch_features<<<grid_for(P, kSkFeatWarps), kSkFeatWarps * 32, smem, s>>>(
      hops, num_nodes, num_perm, hll_p, reinterpret_cast<const uint32_t*>(minhash), hll, u, s_u, v, s_v, P, out,
      reinterpret_cast<unsigned long long*>(info));
  TW_LAUNCH_CHECK();
  return 0;
}
