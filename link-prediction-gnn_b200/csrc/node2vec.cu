// node2vec.cu - node2vec on the device: second-order biased random walks, one skip-gram step with negative sampling and lazy
// (sparse) Adam, and the embedding's pair scores.
//   twowl_n2v_walks       one thread per walk. The next node is proposed uniformly from N(cur) and accepted with probability
//                         w(x) / max(w) (KnightKing's rejection sampling; no alias tables): w = 1/p for the return to prev, 1 for
//                         x in N(prev) (a binary search of prev's sorted list, only when the accept draw falls between the two
//                         thresholds it separates), 1/q otherwise. Every draw is hash_u32 of (walk index, step, trial, draw).
//   twowl_n2v_step        one warp per token: the dots and loss coefficients of its <= window + K pairs; the (row, entry) list of
//                         both ends of every pair, stably radix-sorted by row; one warp per distinct row sums its gradient in
//                         sorted order from the pre-step table, then one warp per row applies SparseAdam. Integer atomics only.
//   twowl_embedding_dot   one warp per pair, the step's dot routine.
// Every result is bitwise repeatable: no floating-point atomics, fixed reduction trees, fixed-order double sums.
#include "common.cuh"

namespace twowl {

constexpr int kN2vWalkThreads = 128;
constexpr int kN2vThreads = 256;
constexpr int kN2vWarps = kN2vThreads / 32;
constexpr int kN2vLossThreads = 1024;
constexpr int kN2vMaxDim = 512;
constexpr int64_t kN2vMaxLength = 1 << 24;          // steps of a walk: 24 bits of the per-step counter
constexpr int64_t kN2vMaxWalkIndex = 1LL << 40;     // walk indices: the other 40 bits
constexpr double kN2vMaxRatio = 1024.0;             // max(w) / min(w): the expected number of trials per step

// the 64-bit key of (walk g, step t): two hashes of the counter g * 2^24 + t; the draws of the step are hash_u32(key, 2 * trial + j)
__device__ __forceinline__ uint64_t n2v_step_key(uint64_t seed, uint64_t g, uint64_t t) {
  const uint64_t c = (g << 24) | t;
  return ((uint64_t)hash_u32(seed, c) << 32) | hash_u32(seed ^ 0xA0761D6478BD642Full, c);
}
// uniform over [0, d) by a 32-bit multiply-high: the bias of any outcome is at most d / 2^32
__device__ __forceinline__ int64_t n2v_uniform(uint32_t h, int64_t d) { return (int64_t)(((uint64_t)h * (uint64_t)d) >> 32); }

__device__ __forceinline__ bool n2v_has(const int32_t* __restrict__ a, int64_t n, int32_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(a + mid) < x) lo = mid + 1;
    else hi = mid;
  }
  return lo < n && __ldg(a + lo) == x;
}

// thr_*: acceptance thresholds on the 32-bit accept draw, floor(w / max(w) * 2^32), 2^32 for the largest weight (always taken)
__global__ void __launch_bounds__(kN2vWalkThreads) k_n2v_walks(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t n,
                                                               const int64_t* __restrict__ start, int64_t s_start, int64_t W, int64_t length,
                                                               uint64_t thr_ret, uint64_t thr_in, uint64_t thr_out, int biased,
                                                               uint64_t seed, int64_t index_base, int32_t* __restrict__ walks) {
  const uint64_t thr_lo = thr_in < thr_out ? thr_in : thr_out, thr_hi = thr_in < thr_out ? thr_out : thr_in;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < W; i += (int64_t)gridDim.x * blockDim.x) {
    int32_t* w = walks + i * length;
    const int64_t s = start[i * s_start];
    const uint64_t g = (uint64_t)(index_base + i);
    const bool ok = s >= 0 && s < n;
    w[0] = ok ? (int32_t)s : -1;
    int64_t prev = -1, cur = ok ? s : -1;
    for (int64_t t = 1; t < length; ++t) {
      int64_t b = 0, d = 0;
      if (cur >= 0) b = ptr[cur], d = ptr[cur + 1] - b;
      if (d == 0) {                       // an isolated start (an undirected walk cannot get stuck anywhere else)
        w[t] = -1;
        cur = -1;
        continue;
      }
      const uint64_t key = n2v_step_key(seed, g, (uint64_t)t);
      int32_t x;
      for (uint32_t trial = 0;; ++trial) {
        x = __ldg(adj + b + n2v_uniform(hash_u32(key, 2ull * trial), d));
        if (!biased || prev < 0) break;
        const uint64_t h = hash_u32(key, 2ull * trial + 1);
        bool acc;
        if (x == prev) acc = h < thr_ret;
        else if (h < thr_lo) acc = true;
        else if (h >= thr_hi) acc = false;
        else acc = h < (n2v_has(adj + ptr[prev], ptr[prev + 1] - ptr[prev], x) ? thr_in : thr_out);
        if (acc) break;
      }
      w[t] = x;
      prev = cur;
      cur = x;
    }
  }
}

// ---------------------------------------------------------------- skip-gram step ---------------------
struct N2vShape {
  int64_t B, L, window, K, n;
  int d;
  __host__ __device__ int64_t tokens() const { return B * L; }
  __host__ __device__ int64_t slots() const { return B * L * (window + K); }
};

// the two rows of pair slot `slot` (slot % S < window: the positive (walks[b, i], walks[b, i + o + 1]), else the negative
// (walks[b, i], negs[b, i, o - window])); false when the slot holds no pair. An id outside [0, n) counts as padding.
__device__ __forceinline__ bool n2v_pair(const int32_t* __restrict__ walks, const int32_t* __restrict__ negs, const N2vShape& sh,
                                         int64_t slot, bool token_active, int32_t& a, int32_t& b) {
  const int64_t S = sh.window + sh.K, tok = slot / S, o = slot - tok * S, i = tok % sh.L;
  a = __ldg(walks + tok);
  if (a < 0 || a >= sh.n) return false;
  if (o < sh.window) {
    if (i + o + 1 >= sh.L) return false;
    b = __ldg(walks + tok + o + 1);
  } else {
    if (!token_active) return false;
    b = __ldg(negs + tok * sh.K + (o - sh.window));
  }
  return b >= 0 && b < sh.n;
}

// positive pairs of token tok
__device__ __forceinline__ int n2v_npos(const int32_t* __restrict__ walks, const N2vShape& sh, int64_t tok) {
  const int32_t a = __ldg(walks + tok);
  if (a < 0 || a >= sh.n) return 0;
  const int64_t i = tok % sh.L;
  int c = 0;
  for (int64_t o = 1; o <= sh.window && i + o < sh.L; ++o) {
    const int32_t b = __ldg(walks + tok + o);
    c += b >= 0 && b < sh.n;
  }
  return c;
}

// e_a . e_b over d = 32 * nc elements: lane l adds elements l, l + 32, ... in order with fma, then an xor butterfly. Every lane
// ends with the same value, and dot(a, b) == dot(b, a) bit for bit.
__device__ __forceinline__ float n2v_dot(const float* __restrict__ ea, const float* __restrict__ eb, int nc, int lane) {
  float s = 0.f;
  for (int c = 0; c < nc; ++c) s = fmaf(__ldg(ea + c * 32 + lane), __ldg(eb + c * 32 + lane), s);
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
  return s;
}

__device__ __forceinline__ double softplus_d(double x) { return fmax(x, 0.0) + log1p(exp(-fabs(x))); }

// cnt[0] = positive pairs, cnt[1] = tokens with at least one
__global__ void __launch_bounds__(kN2vThreads) k_n2v_count(const int32_t* __restrict__ walks, N2vShape sh,
                                                           unsigned long long* __restrict__ cnt) {
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < sh.tokens(); base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t tok = base + threadIdx.x;
    const unsigned c = tok < sh.tokens() ? (unsigned)n2v_npos(walks, sh, tok) : 0u;
    const unsigned sc = __reduce_add_sync(0xffffffffu, c), sa = __reduce_add_sync(0xffffffffu, c > 0 ? 1u : 0u);
    if ((threadIdx.x & 31) == 0 && sc) {
      atomicAdd(cnt, (unsigned long long)sc);
      atomicAdd(cnt + 1, (unsigned long long)sa);
    }
  }
}

// one warp per token: coef[slot] = d loss / d (e_a . e_b), the entries (row, 2 slot + end) of both ends, the token's loss sums
__global__ void __launch_bounds__(kN2vThreads) k_n2v_pairs(const float* __restrict__ emb, const int32_t* __restrict__ walks,
                                                           const int32_t* __restrict__ negs, N2vShape sh,
                                                           const unsigned long long* __restrict__ cnt, float* __restrict__ coef,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                           double* __restrict__ loss_pos, double* __restrict__ loss_neg) {
  const int lane = threadIdx.x & 31, nc = sh.d / 32;
  const int64_t S = sh.window + sh.K;
  const double npos = (double)cnt[0], nneg = (double)cnt[1] * (double)sh.K;
  for (int64_t tok = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; tok < sh.tokens(); tok += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const bool active = n2v_npos(walks, sh, tok) > 0;
    double lp = 0.0, ln = 0.0;
    for (int64_t o = 0; o < S; ++o) {
      const int64_t slot = tok * S + o;
      int32_t a, b;
      const bool ok = n2v_pair(walks, negs, sh, slot, active, a, b);
      float c = 0.f;
      if (ok) {
        const double x = (double)n2v_dot(emb + (int64_t)a * sh.d, emb + (int64_t)b * sh.d, nc, lane);
        const double e = exp(-fabs(x));
        const double sig = x >= 0 ? 1.0 / (1.0 + e) : e / (1.0 + e), sig_neg = x >= 0 ? e / (1.0 + e) : 1.0 / (1.0 + e);
        if (o < sh.window) {
          lp += softplus_d(-x);
          c = (float)(-sig_neg / npos);           // d softplus(-x) / dx = sigma(x) - 1 = -sigma(-x)
        } else {
          ln += softplus_d(x);
          c = (float)(sig / nneg);
        }
      }
      if (lane == 0) {
        coef[slot] = c;
        keys[2 * slot] = ok ? (uint32_t)a : (uint32_t)sh.n;
        keys[2 * slot + 1] = ok ? (uint32_t)b : (uint32_t)sh.n;
        vals[2 * slot] = (uint32_t)(2 * slot);
        vals[2 * slot + 1] = (uint32_t)(2 * slot + 1);
      }
    }
    if (lane == 0) loss_pos[tok] = lp, loss_neg[tok] = ln;
  }
}

// head[i] = 1 where a run of equal rows starts in the sorted keys (rows < n only)
__global__ void __launch_bounds__(kN2vThreads) k_n2v_heads(const uint32_t* __restrict__ keys, int64_t E, uint32_t n, int64_t* __restrict__ head) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = keys[i];
    head[i] = k < n && (i == 0 || keys[i - 1] != k);
  }
}

// seg_start[u] = the first entry of distinct row u; seg_start[U] = the number of entries with a row
__global__ void __launch_bounds__(kN2vThreads) k_n2v_starts(const uint32_t* __restrict__ keys, int64_t E, uint32_t n,
                                                            const int64_t* __restrict__ head, int64_t* __restrict__ seg_start) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < E; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = keys[i];
    if (k >= n) continue;
    if (i == 0 || keys[i - 1] != k) seg_start[head[i]] = i;
    if (i == E - 1 || keys[i + 1] >= n) seg_start[head[E]] = i + 1;
  }
}

// one warp per distinct row: G[u] = sum over its entries, in sorted (= entry) order, of coef * e_other, from the pre-step table
__global__ void __launch_bounds__(kN2vThreads) k_n2v_grad(const float* __restrict__ emb, const int32_t* __restrict__ walks,
                                                          const int32_t* __restrict__ negs, N2vShape sh, const uint32_t* __restrict__ vals,
                                                          const float* __restrict__ coef, const int64_t* __restrict__ head, int64_t E,
                                                          const int64_t* __restrict__ seg_start, float* __restrict__ G) {
  const int lane = threadIdx.x & 31, nc = sh.d / 32;
  const int64_t U = head[E];
  for (int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < U; u += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    float g[kN2vMaxDim / 32];
#pragma unroll
    for (int c = 0; c < kN2vMaxDim / 32; ++c) g[c] = 0.f;
    const int64_t j1 = seg_start[u + 1];
    for (int64_t j = seg_start[u]; j < j1; ++j) {
      const uint32_t e = __ldg(vals + j);
      const int64_t slot = e >> 1;
      int32_t a, b;
      n2v_pair(walks, negs, sh, slot, true, a, b);   // a valid slot: its rows do not depend on the token's activity
      const float* eo = emb + (int64_t)((e & 1) ? a : b) * sh.d;
      const float c0 = __ldg(coef + slot);
#pragma unroll
      for (int c = 0; c < kN2vMaxDim / 32; ++c)
        if (c < nc) g[c] = fmaf(c0, __ldg(eo + c * 32 + lane), g[c]);
    }
#pragma unroll
    for (int c = 0; c < kN2vMaxDim / 32; ++c)
      if (c < nc) G[u * sh.d + c * 32 + lane] = g[c];
  }
}

// torch.optim.SparseAdam on each distinct row: m += (g - m)(1 - b1), v += (g^2 - v)(1 - b2),
// p -= lr sqrt(1 - b2^t) / (1 - b1^t) * m / (sqrt(v) + eps), t = step[0] + 1. The scalars are formed in double from the double
// hyper-parameters and rounded to fp32 where they meet the tensors, as torch does: 1 - 0.999f in fp32 would be 4.7e-5 off.
__global__ void __launch_bounds__(kN2vThreads) k_n2v_adam(float* __restrict__ emb, float* __restrict__ m, float* __restrict__ v, int d,
                                                          const uint32_t* __restrict__ keys, const int64_t* __restrict__ head, int64_t E,
                                                          const int64_t* __restrict__ seg_start, const float* __restrict__ G, double lr,
                                                          double beta1, double beta2, double eps, const int64_t* __restrict__ step) {
  const int64_t U = head[E];
  const int64_t t = step[0] + 1;
  const double bc1 = 1.0 - pow(beta1, (double)t), bc2 = 1.0 - pow(beta2, (double)t);
  const float step_size = (float)(lr * sqrt(bc2) / bc1);
  const float w1 = (float)(1.0 - beta1), w2 = (float)(1.0 - beta2), epsf = (float)eps;
  const int lane = threadIdx.x & 31;
  for (int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < U; u += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int64_t row = keys[seg_start[u]];
    for (int c = lane; c < d; c += 32) {
      const int64_t k = row * d + c;
      const float g = G[u * d + c], m0 = m[k], v0 = v[k];
      const float mi = m0 + (g - m0) * w1;
      const float vi = v0 + (g * g - v0) * w2;
      m[k] = mi, v[k] = vi;
      emb[k] -= step_size * (mi / (sqrtf(vi) + epsf));
    }
  }
}

// loss = sum(loss_pos) / npos + sum(loss_neg) / nneg, each a fixed-order double sum (0 without a positive pair); step += 1 if any
__global__ void __launch_bounds__(kN2vLossThreads) k_n2v_finish(const double* __restrict__ loss_pos, const double* __restrict__ loss_neg,
                                                                int64_t T, int64_t K, const unsigned long long* __restrict__ cnt,
                                                                double* __restrict__ loss, int64_t* __restrict__ step) {
  __shared__ double sp[kN2vLossThreads], sn[kN2vLossThreads];
  const int64_t per = (T + kN2vLossThreads - 1) / kN2vLossThreads, b = (int64_t)threadIdx.x * per, e = b + per < T ? b + per : T;
  double p = 0.0, q = 0.0;
  for (int64_t i = b; i < e; ++i) p += loss_pos[i], q += loss_neg[i];
  sp[threadIdx.x] = p, sn[threadIdx.x] = q;
  __syncthreads();
  for (int h = kN2vLossThreads / 2; h > 0; h >>= 1) {
    if ((int)threadIdx.x < h) sp[threadIdx.x] += sp[threadIdx.x + h], sn[threadIdx.x] += sn[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const unsigned long long np = cnt[0];
    loss[0] = np ? sp[0] / (double)np + sn[0] / ((double)cnt[1] * (double)K) : 0.0;
    if (np) step[0] += 1;
  }
}

__global__ void __launch_bounds__(kN2vThreads) k_embedding_dot(const float* __restrict__ emb, int64_t n, int d, const int64_t* __restrict__ u,
                                                               int64_t s_u, const int64_t* __restrict__ v, int64_t s_v, int64_t P,
                                                               float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < P; i += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int64_t a = u[i * s_u], b = v[i * s_v];
    const bool ok = a >= 0 && a < n && b >= 0 && b < n;
    const float s = ok ? n2v_dot(emb + a * d, emb + b * d, d / 32, lane) : __int_as_float(0x7fffffff);
    if (lane == 0) out[i] = s;
  }
}

struct N2vWs {
  unsigned long long* cnt;
  float* coef;
  double *loss_pos, *loss_neg;
  uint32_t *k0, *v0, *k1, *v1;
  void* rws;
  int64_t *head, *seg_start;
  void* sws;
  float* G;
};

// the workspace of twowl_n2v_step laid out from `base` (NULL: only its size is wanted). A distinct row is a token or a negative,
// so there are at most B L (1 + K) of them.
static size_t n2v_step_carve(void* base, int64_t B, int64_t L, int64_t window, int64_t K, int64_t d, N2vWs& w) {
  const int64_t T = B * L, slots = T * (window + K), E = 2 * slots, U = T * (1 + K);
  Carver c(base);
  w.cnt = c.take<unsigned long long>(2);
  w.coef = c.take<float>(slots);
  w.loss_pos = c.take<double>(T);
  w.loss_neg = c.take<double>(T);
  w.k0 = c.take<uint32_t>(E);
  w.v0 = c.take<uint32_t>(E);
  w.k1 = c.take<uint32_t>(E);
  w.v1 = c.take<uint32_t>(E);
  w.rws = c.take<char>(radix_workspace_bytes(E));
  w.head = c.take<int64_t>(E + 1);
  w.seg_start = c.take<int64_t>(U + 1);
  w.sws = c.take<char>(scan_workspace_bytes(E));
  w.G = c.take<float>(U * d);
  return c.off;
}

static bool n2v_dim_ok(int64_t d) { return d >= 32 && d <= kN2vMaxDim && d % 32 == 0; }

}  // namespace twowl

using namespace twowl;

extern "C" int twowl_n2v_walks(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, const int64_t* start, int64_t s_start, int64_t W,
                               int64_t length, float p, float q, uint64_t seed, int64_t index_base, int32_t* walks, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && W >= 0 && length >= 1 && length <= kN2vMaxLength && index_base >= 0 &&
                   index_base + W <= kN2vMaxWalkIndex && W * length < (1LL << 62),
               "n2v_walks: bad sizes (W >= 0, 1 <= length <= 2^24, 0 <= index_base, index_base + W <= 2^40)");
  const double wr = 1.0 / (double)p, wo = 1.0 / (double)q;
  const double wmax = fmax(fmax(wr, 1.0), wo), wmin = fmin(fmin(wr, 1.0), wo);
  TW_CHECK_ARG(p > 0.f && q > 0.f && p <= 3.4e38f && q <= 3.4e38f && wmax / wmin <= kN2vMaxRatio,
               "n2v_walks: p and q must be finite and > 0, with max(1/p, 1, 1/q) / min(1/p, 1, 1/q) <= 1024");
  TW_CHECK_ARG(W == 0 || (ptr && start && walks), "n2v_walks: null pointer");   // adj: NULL when nnz = 0
  if (W == 0) return 0;
  auto thr = [&](double w) { return w >= wmax ? (1ull << 32) : (uint64_t)(w / wmax * 4294967296.0); };
  const int biased = !(p == 1.f && q == 1.f);
  k_n2v_walks<<<grid_for(W, kN2vWalkThreads), kN2vWalkThreads, 0, (cudaStream_t)stream>>>(
      ptr, adj, num_nodes, start, s_start, W, length, thr(wr), thr(1.0), thr(wo), biased, seed, index_base, walks);
  TW_LAUNCH_CHECK();
  return 0;
}

static bool n2v_step_sizes_ok(int64_t B, int64_t L, int64_t window, int64_t K) {
  return B >= 0 && L >= 0 && B < (1LL << 31) && L < (1LL << 31) && window >= 1 && K >= 1 && window < (1LL << 20) && K < (1LL << 20) &&
         B * L < (1LL << 31) && 2 * B * L * (window + K) < 0x80000000LL;
}

extern "C" size_t twowl_n2v_step_workspace_bytes(int64_t B, int64_t L, int64_t window, int64_t K, int64_t d) {
  if (!n2v_step_sizes_ok(B, L, window, K) || !n2v_dim_ok(d)) return 0;
  N2vWs w;
  return n2v_step_carve(nullptr, B, L, window, K, d, w);
}

extern "C" int twowl_n2v_step(float* emb, float* exp_avg, float* exp_avg_sq, int64_t* step, int64_t num_nodes, int32_t d,
                              const int32_t* walks, const int32_t* negs, int64_t B, int64_t L, int64_t window, int64_t K, double lr,
                              double beta1, double beta2, double eps, double* loss, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && n2v_step_sizes_ok(B, L, window, K),
               "n2v_step: bad sizes (B, L >= 0, window >= 1, K >= 1, 2 B L (window + K) < 2^31)");
  TW_CHECK_ARG(n2v_dim_ok(d), "n2v_step: d must be a multiple of 32 in [32, 512]");
  TW_CHECK_ARG(lr >= 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0, "n2v_step: bad hyper-parameters");
  TW_CHECK_ARG(step && loss && (B * L == 0 || (walks && negs)) && (num_nodes == 0 || (emb && exp_avg && exp_avg_sq)),
               "n2v_step: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_n2v_step_workspace_bytes(B, L, window, K, d));
  cudaStream_t s = (cudaStream_t)stream;
  N2vWs w;
  n2v_step_carve(ws, B, L, window, K, d, w);
  const N2vShape sh{B, L, window, K, num_nodes, d};
  const int64_t T = sh.tokens(), E = 2 * sh.slots(), Umax = T * (1 + K);
  TW_CUDA(cudaMemsetAsync(w.cnt, 0, 2 * sizeof(unsigned long long), s));
  if (T > 0) {
    k_n2v_count<<<grid_for(T, kN2vThreads), kN2vThreads, 0, s>>>(walks, sh, w.cnt);
    k_n2v_pairs<<<grid_for(T, kN2vWarps), kN2vThreads, 0, s>>>(emb, walks, negs, sh, w.cnt, w.coef, w.k0, w.v0, w.loss_pos, w.loss_neg);
    TW_LAUNCH_CHECK();
    // stably by row: each row's entries stay in entry order, the order its gradient is summed in; no row (key n) sorts last
    if (int rc = radix_sort_pairs(w.k0, w.v0, w.k1, w.v1, E, bits_for_value(num_nodes), w.rws, s)) return rc;
    k_n2v_heads<<<grid_for(E, kN2vThreads), kN2vThreads, 0, s>>>(w.k1, E, (uint32_t)num_nodes, w.head);
    TW_LAUNCH_CHECK();
    if (int rc = scan_exclusive_i64(w.head, w.head, E, w.sws, s)) return rc;
    k_n2v_starts<<<grid_for(E, kN2vThreads), kN2vThreads, 0, s>>>(w.k1, E, (uint32_t)num_nodes, w.head, w.seg_start);
    k_n2v_grad<<<grid_for(Umax, kN2vWarps), kN2vThreads, 0, s>>>(emb, walks, negs, sh, w.v1, w.coef, w.head, E, w.seg_start, w.G);
    k_n2v_adam<<<grid_for(Umax, kN2vWarps), kN2vThreads, 0, s>>>(emb, exp_avg, exp_avg_sq, d, w.k1, w.head, E, w.seg_start, w.G, lr, beta1,
                                                                 beta2, eps, step);
    TW_LAUNCH_CHECK();
  }
  k_n2v_finish<<<1, kN2vLossThreads, 0, s>>>(w.loss_pos, w.loss_neg, T, K, w.cnt, loss, step);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_embedding_dot(const float* emb, int64_t num_nodes, int32_t d, const int64_t* u, int64_t s_u, const int64_t* v,
                                   int64_t s_v, int64_t P, float* out, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && P >= 0, "embedding_dot: bad sizes (num_nodes, P >= 0)");
  TW_CHECK_ARG(n2v_dim_ok(d), "embedding_dot: d must be a multiple of 32 in [32, 512]");
  TW_CHECK_ARG(P == 0 || (u && v && out && (num_nodes == 0 || emb)), "embedding_dot: null pointer");
  if (P == 0) return 0;
  k_embedding_dot<<<grid_for(P, kN2vWarps), kN2vThreads, 0, (cudaStream_t)stream>>>(emb, num_nodes, d, u, s_u, v, s_v, P, out);
  TW_LAUNCH_CHECK();
  return 0;
}
