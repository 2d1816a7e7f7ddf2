// metrics.cu - ROC-AUC on the device, replacing the per-step host round trip of the reference's train / test loop
// (TwoWL/model/train.py:41-43 and :61-66: pred.sigmoid().cpu().numpy() -> sklearn.metrics.roc_auc_score).
//
// AUC = (sum of the average ranks of the positives - n_pos (n_pos + 1) / 2) / (n_pos n_neg)   (Mann-Whitney U with ties
// sharing their average rank = the area under the trapezoidal ROC curve sklearn integrates). Scores are sorted with the
// library's stable LSD radix sort on an order-preserving 32-bit key; each element finds its tie group by binary search
// in the sorted keys; sums are integer / double with a fixed two-level order: deterministic, no atomics.
//
// Ranking metrics of the OGB link-prediction evaluators (ogb/linkproppred/evaluate.py):
//   hits@K against a shared negative set (_eval_hits: ogbl-collab, ogbl-ddi) - the same key / radix sort as the AUC with every
//     positive's key forced to 0, which no non-NaN score maps to: the negatives sort on top, the K-th largest negative sits at
//     sorted position n - K, and a second pass counts the positives strictly above it. Integer counts: deterministic.
//   MRR and hits@k against k negatives per positive (_eval_mrr: ogbl-citation2) - one warp per row counts the negatives above
//     (optimistic) and at-or-above (pessimistic) its positive; 1 / rank is summed in double in a fixed two-level order.
#include "common.cuh"

namespace twowl {

constexpr int kAucThreads = 256;
constexpr int kAucMaxCtas = kNumSMs * 4;

__device__ __forceinline__ uint32_t auc_key(float x) {
  // ascending order-preserving map of IEEE-754 floats to uint32 (-0 and +0 share a key; NaNs sort last)
  if (x == 0.f) x = 0.f;
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(kAucThreads) k_auc_keys(const float* __restrict__ score, int64_t n, uint32_t* __restrict__ keys,
                                                          uint32_t* __restrict__ vals) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = auc_key(score[i]);
    vals[i] = (uint32_t)i;
  }
}

// per CTA: (sum over positives of 2 * average rank, number of positives) as (double, int64)
__global__ void __launch_bounds__(kAucThreads) k_auc_ranks(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                           const float* __restrict__ label, int64_t n, double* __restrict__ part) {
  __shared__ double s_r[kAucThreads];
  __shared__ double s_p[kAucThreads];
  double r2 = 0, np = 0;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    if (!(label[vals[j]] > 0.5f)) continue;
    const uint32_t k = keys[j];
    int64_t lo = 0, hi = j;          // first position with key == k
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] < k) lo = mid + 1; else hi = mid;
    }
    const int64_t s = lo;
    lo = j + 1, hi = n;               // first position with key > k
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (keys[mid] <= k) lo = mid + 1; else hi = mid;
    }
    r2 += (double)(s + lo + 1);       // ranks s+1 .. lo: twice their average
    np += 1.0;
  }
  s_r[threadIdx.x] = r2, s_p[threadIdx.x] = np;
  __syncthreads();
  for (int d = kAucThreads / 2; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) s_r[threadIdx.x] += s_r[threadIdx.x + d], s_p[threadIdx.x] += s_p[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[2 * blockIdx.x] = s_r[0], part[2 * blockIdx.x + 1] = s_p[0];
}

__global__ void k_auc_final(const double* __restrict__ part, int nparts, int64_t n, double* __restrict__ out) {
  double r2 = 0, np = 0;
  for (int b = 0; b < nparts; ++b) r2 += part[2 * b], np += part[2 * b + 1];
  const double nn = (double)n - np;
  out[1] = np, out[2] = nn;
  out[0] = (np > 0 && nn > 0) ? (0.5 * r2 - 0.5 * np * (np + 1.0)) / (np * nn) : nan("");
}

// ---- ranking metrics -------------------------------------------------------------------------------------------------------
constexpr int kRankMaxK = TWOWL_RANK_MAX_K;   // cut-offs per call
struct RankKs {                      // the host's cut-off list, passed by value
  int64_t k[kRankMaxK];
};

// keys[i] = 0 for a positive, the order-preserving key of its score for a negative; any NaN score raises *nan_flag
__global__ void __launch_bounds__(kAucThreads) k_hits_keys(const float* __restrict__ score, const float* __restrict__ label, int64_t n,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ vals, int* __restrict__ nan_flag) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float x = score[i];
    if (isnan(x)) *nan_flag = 1;
    keys[i] = label[i] > 0.5f ? 0u : auc_key(x);
    vals[i] = (uint32_t)i;
  }
}

// cnt[j] += #(positives with key > kth_j), cnt[n_k] += #positives. kth_j = the sorted key at n - K_j, or 0 when it is a positive's
// (fewer than K_j negatives): every non-NaN key is above 0, so every positive counts and hits@K_j = 1, OGB's rule.
__global__ void __launch_bounds__(kAucThreads) k_hits_count(const float* __restrict__ score, const float* __restrict__ label, int64_t n,
                                                            const uint32_t* __restrict__ sorted, RankKs ks, int n_k,
                                                            unsigned long long* __restrict__ cnt) {
  uint32_t thr[kRankMaxK];
  unsigned c[kRankMaxK + 1];
#pragma unroll
  for (int j = 0; j < kRankMaxK; ++j) {
    thr[j] = (j < n_k && ks.k[j] <= n) ? sorted[n - ks.k[j]] : 0u;
    c[j] = 0;
  }
  c[kRankMaxK] = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!(label[i] > 0.5f)) continue;
    const uint32_t key = auc_key(score[i]);
    c[kRankMaxK] += 1;
#pragma unroll
    for (int j = 0; j < kRankMaxK; ++j) c[j] += key > thr[j];
  }
  const int lane = threadIdx.x & 31;
  const unsigned np = __reduce_add_sync(0xffffffffu, c[kRankMaxK]);
  if (lane == 0 && np) atomicAdd(cnt + n_k, (unsigned long long)np);
#pragma unroll
  for (int j = 0; j < kRankMaxK; ++j) {
    const unsigned h = __reduce_add_sync(0xffffffffu, c[j]);
    if (j < n_k && lane == 0 && h) atomicAdd(cnt + j, (unsigned long long)h);
  }
}

__global__ void k_hits_final(const unsigned long long* __restrict__ cnt, const int* __restrict__ nan_flag, int n_k, int64_t n,
                             double* __restrict__ out) {
  const double np = (double)cnt[n_k];
  const bool bad = *nan_flag || np == 0;
  for (int j = 0; j < n_k; ++j) out[j] = bad ? nan("") : (double)cnt[j] / np;
  out[n_k] = np, out[n_k + 1] = (double)n - np;
}

constexpr int kRankThreads = 256;
constexpr int kRankWarps = kRankThreads / 32;

// one warp per row i: opt = #(neg_ij > pos_i), pess = #(neg_ij >= pos_i), 2 rank = opt + pess + 2. Per CTA: the sum of 1 / rank
// (each warp over its rows in order, then the warps in order) and hits counts #(2 rank <= 2 k_j).
__global__ void __launch_bounds__(kRankThreads) k_rank_rows(const float* __restrict__ pos, const float* __restrict__ neg, int64_t P,
                                                            int64_t k, RankKs ks, int n_k, double* __restrict__ part_rr,
                                                            unsigned long long* __restrict__ part_hits, int* __restrict__ nan_flag) {
  __shared__ double s_rr[kRankWarps];
  __shared__ unsigned s_hits[kRankWarps][kRankMaxK];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double rr = 0;
  unsigned hits[kRankMaxK];
#pragma unroll
  for (int j = 0; j < kRankMaxK; ++j) hits[j] = 0;
  bool nan_seen = false;
  for (int64_t i = (int64_t)blockIdx.x * kRankWarps + warp; i < P; i += (int64_t)gridDim.x * kRankWarps) {
    const float p = pos[i];
    const float* row = neg + i * k;
    unsigned opt = 0, pess = 0;
    bool bad = isnan(p);
#pragma unroll 4
    for (int64_t j = lane; j < k; j += 32) {
      const float v = __ldg(row + j);
      opt += v > p;
      pess += v >= p;
      bad |= isnan(v);
    }
    opt = __reduce_add_sync(0xffffffffu, opt);
    pess = __reduce_add_sync(0xffffffffu, pess);
    nan_seen |= bad;
    const int64_t rank2 = (int64_t)opt + pess + 2;
    rr += 2.0 / (double)rank2;
#pragma unroll
    for (int j = 0; j < kRankMaxK; ++j) hits[j] += rank2 <= 2 * ks.k[j];
  }
  if (__any_sync(0xffffffffu, nan_seen) && lane == 0) *nan_flag = 1;
  if (lane == 0) {
    s_rr[warp] = rr;
#pragma unroll
    for (int j = 0; j < kRankMaxK; ++j) s_hits[warp][j] = hits[j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < kRankWarps; ++w) t += s_rr[w];
    part_rr[blockIdx.x] = t;
  }
  if ((int)threadIdx.x < n_k) {
    unsigned long long h = 0;
    for (int w = 0; w < kRankWarps; ++w) h += s_hits[w][threadIdx.x];
    part_hits[(int64_t)blockIdx.x * n_k + threadIdx.x] = h;
  }
}

__global__ void k_rank_final(const double* __restrict__ part_rr, const unsigned long long* __restrict__ part_hits, int nparts,
                             const int* __restrict__ nan_flag, int n_k, int64_t P, double* __restrict__ out) {
  const bool bad = *nan_flag || P == 0;
  double rr = 0;
  for (int b = 0; b < nparts; ++b) rr += part_rr[b];
  out[0] = bad ? nan("") : rr / (double)P;
  for (int j = 0; j < n_k; ++j) {
    unsigned long long h = 0;
    for (int b = 0; b < nparts; ++b) h += part_hits[(int64_t)b * n_k + j];
    out[1 + j] = bad ? nan("") : (double)h / (double)P;
  }
  out[n_k + 1] = (double)P;
}

static bool rank_ks(const int64_t* h_ks, int n_k, RankKs* ks) {
  if (!h_ks || n_k < 1 || n_k > kRankMaxK) return false;
  for (int j = 0; j < kRankMaxK; ++j) {
    ks->k[j] = j < n_k ? h_ks[j] : 1;
    if (ks->k[j] < 1) return false;
  }
  return true;
}

static int rank_grid(int64_t P) { return grid_for(P, kRankWarps, 8); }

}  // namespace twowl

using namespace twowl;

extern "C" size_t twowl_auc_workspace_bytes(int64_t n) {
  const size_t m = (size_t)(n > 0 ? n : 1);
  return 4 * align_up(m * sizeof(uint32_t)) + align_up(radix_workspace_bytes(n)) + align_up((size_t)kAucMaxCtas * 2 * sizeof(double));
}

extern "C" int twowl_auc(const float* score, const float* label, int64_t n, double* out, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(n >= 0 && n < 0x7fffffffLL, "auc: n out of range");
  TW_CHECK_ARG(score && label && out, "auc: null pointer");
  TW_CHECK_WS(ws_bytes, twowl_auc_workspace_bytes(n));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t m = (size_t)(n > 0 ? n : 1);
  Carver c(ws);
  uint32_t* k0 = c.take<uint32_t>(m);
  uint32_t* v0 = c.take<uint32_t>(m);
  uint32_t* k1 = c.take<uint32_t>(m);
  uint32_t* v1 = c.take<uint32_t>(m);
  void* rws = c.take<char>(radix_workspace_bytes(n));
  double* part = c.take<double>((size_t)kAucMaxCtas * 2);
  const int grid = n > 0 ? grid_for(n, kAucThreads, 4) : 1;
  if (n > 0) {
    k_auc_keys<<<grid, kAucThreads, 0, s>>>(score, n, k0, v0);
    TW_LAUNCH_CHECK();
    if (int rc = radix_sort_pairs(k0, v0, k1, v1, n, 32, rws, s)) return rc;
  }
  k_auc_ranks<<<grid, kAucThreads, 0, s>>>(k1, v1, label, n, part);
  k_auc_final<<<1, 1, 0, s>>>(part, grid, n, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_hits_at_k_workspace_bytes(int64_t n) {
  const size_t m = (size_t)(n > 0 ? n : 1);
  return 4 * align_up(m * sizeof(uint32_t)) + align_up(radix_workspace_bytes(n)) +
         align_up((kRankMaxK + 1) * sizeof(unsigned long long)) + align_up(sizeof(int));
}

extern "C" int twowl_hits_at_k(const float* score, const float* label, int64_t n, const int64_t* h_ks, int32_t n_k, double* out,
                               void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(n >= 0 && n < 0x7fffffffLL, "hits_at_k: n out of range");
  TW_CHECK_ARG(out && (n == 0 || (score && label)), "hits_at_k: null pointer");
  RankKs ks;
  TW_CHECK_ARG(rank_ks(h_ks, n_k, &ks), "hits_at_k: ks must hold 1..%d values, each >= 1", kRankMaxK);
  TW_CHECK_WS(ws_bytes, twowl_hits_at_k_workspace_bytes(n));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t m = (size_t)(n > 0 ? n : 1);
  Carver c(ws);
  uint32_t* k0 = c.take<uint32_t>(m);
  uint32_t* v0 = c.take<uint32_t>(m);
  uint32_t* k1 = c.take<uint32_t>(m);
  uint32_t* v1 = c.take<uint32_t>(m);
  void* rws = c.take<char>(radix_workspace_bytes(n));
  unsigned long long* cnt = c.take<unsigned long long>(kRankMaxK + 1);
  int* nan_flag = c.take<int>(1);
  TW_CUDA(cudaMemsetAsync(cnt, 0, (kRankMaxK + 1) * sizeof(unsigned long long), s));
  TW_CUDA(cudaMemsetAsync(nan_flag, 0, sizeof(int), s));
  if (n > 0) {
    const int grid = grid_for(n, kAucThreads, 4);
    k_hits_keys<<<grid, kAucThreads, 0, s>>>(score, label, n, k0, v0, nan_flag);
    TW_LAUNCH_CHECK();
    if (int rc = radix_sort_pairs(k0, v0, k1, v1, n, 32, rws, s)) return rc;
    k_hits_count<<<grid, kAucThreads, 0, s>>>(score, label, n, k1, ks, n_k, cnt);
  }
  k_hits_final<<<1, 1, 0, s>>>(cnt, nan_flag, n_k, n, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_rank_metrics_workspace_bytes(int64_t P) {
  const size_t g = (size_t)rank_grid(P);
  return align_up(g * sizeof(double)) + align_up(g * kRankMaxK * sizeof(unsigned long long)) + align_up(sizeof(int));
}

extern "C" int twowl_rank_metrics(const float* pos, const float* neg, int64_t P, int64_t k, const int64_t* h_ks, int32_t n_k,
                                  double* out, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(P >= 0 && k >= 1 && P < 0x7fffffffLL && k < 0x7fffffffLL, "rank_metrics: bad sizes (0 <= P < 2^31, 1 <= k < 2^31)");
  TW_CHECK_ARG(out && (P == 0 || (pos && neg)), "rank_metrics: null pointer");
  RankKs ks;
  TW_CHECK_ARG(rank_ks(h_ks, n_k, &ks), "rank_metrics: ks must hold 1..%d values, each >= 1", kRankMaxK);
  TW_CHECK_WS(ws_bytes, twowl_rank_metrics_workspace_bytes(P));
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = rank_grid(P);
  Carver c(ws);
  double* part_rr = c.take<double>(grid);
  unsigned long long* part_hits = c.take<unsigned long long>((size_t)grid * kRankMaxK);
  int* nan_flag = c.take<int>(1);
  TW_CUDA(cudaMemsetAsync(nan_flag, 0, sizeof(int), s));
  k_rank_rows<<<grid, kRankThreads, 0, s>>>(pos, neg, P, k, ks, n_k, part_rr, part_hits, nan_flag);
  k_rank_final<<<1, 1, 0, s>>>(part_rr, part_hits, grid, nan_flag, n_k, P, out);
  TW_LAUNCH_CHECK();
  return 0;
}
