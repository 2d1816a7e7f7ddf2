// pair_ops.cu - the row-wise gather kernels around the aggregations: nn.Embedding lookup
// (TwoWL/model/model.py:53,71), pair init x[pos[:,0]]*x[pos[:,1]] (model.py:75), readout
// x[idx]; even*odd; Linear(c2,1) (model.py:78-83) and the structured ("factorised") form of the pair-level
// GCNConv for wedge indices that come from get_ei2 + blockei2 (TwoWL/utils.py:36-50).
// All HBM-bound: one lane per float4 of a row, 128-bit accesses, grid-stride over rows.
#include "common.cuh"

namespace twowl {

constexpr int kRowThreads = 256;

// thread -> (row slot, float4 column) map shared by the row kernels (see norm.cu)
struct RowSlots {
  int cv, slots, slot, c4;
  __device__ RowSlots(int C) {
    cv = C >> 2;
    slots = kRowThreads / cv;
    slot = ((int)threadIdx.x < slots * cv) ? (int)threadIdx.x / cv : -1;
    c4 = threadIdx.x % cv;
  }
};

static int row_grid(int64_t rows, int C) {
  const int slots = kRowThreads / (C >> 2);
  return grid_for(rows, slots, 8);
}

__global__ void __launch_bounds__(kRowThreads) k_gather_rows(const float* __restrict__ W, int64_t rows_w,
                                                             const int64_t* __restrict__ idx, int64_t stride, int64_t n, int C,
                                                             float* __restrict__ out) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ W4 = reinterpret_cast<const float4*>(W);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(out);
  for (int64_t r = (int64_t)blockIdx.x * rs.slots + rs.slot; r < n; r += (int64_t)gridDim.x * rs.slots) {
    int64_t s = idx[r * stride];
    if (s < 0) s += rows_w;
    float4 v = f4_zero();
    if (s >= 0 && s < rows_w) v = ldg_cached(W4 + s * rs.cv + rs.c4);
    stg_stream(o4 + r * rs.cv + rs.c4, v);
  }
}

// out[r] = X[src[r << sh]] * X[dst[r << sh]] for r < R (sh = 1: one row per mated pair, see twowl_pair_init_fwd)
__global__ void __launch_bounds__(kRowThreads) k_pair_init(const float* __restrict__ X, const int32_t* __restrict__ src,
                                                           const int32_t* __restrict__ dst, int64_t R, int C, int sh,
                                                           float* __restrict__ out) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(X);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(out);
  for (int64_t r = (int64_t)blockIdx.x * rs.slots + rs.slot; r < R; r += (int64_t)gridDim.x * rs.slots) {
    const float4 a = ldg_cached(X4 + (int64_t)src[r << sh] * rs.cv + rs.c4);
    const float4 b = ldg_cached(X4 + (int64_t)dst[r << sh] * rs.cv + rs.c4);
    stg_stream(o4 + r * rs.cv + rs.c4, f4_mul(a, b));
  }
}

// ---------------------------------------------------------------- readout ------------------------
// one warp per target link l: pred[l] = sum_c H[i0,c]*H[i1,c]*w[c] + b   (xor-shuffle tree, fixed order)
__global__ void __launch_bounds__(kRowThreads) k_readout_fwd(const float* __restrict__ H, const int64_t* __restrict__ idx,
                                                             int64_t sidx, int64_t L, int C, const float* __restrict__ w,
                                                             const float* __restrict__ b, float* __restrict__ pred) {
  const int lane = threadIdx.x & 31;
  const int cv = C >> 2;
  const float4* __restrict__ H4 = reinterpret_cast<const float4*>(H);
  const float4* __restrict__ w4 = reinterpret_cast<const float4*>(w);
  const int64_t warp0 = ((int64_t)blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kRowThreads) >> 5;
  for (int64_t l = warp0; l < L; l += nwarps) {
    const int64_t i0 = idx[(2 * l) * sidx], i1 = idx[(2 * l + 1) * sidx];
    float acc = 0.f;
    for (int c4 = lane; c4 < cv; c4 += 32) {
      const float4 a = ldg_cached(H4 + i0 * cv + c4), c = ldg_cached(H4 + i1 * cv + c4), ww = __ldg(w4 + c4);
      acc = fmaf(a.x * c.x, ww.x, acc);
      acc = fmaf(a.y * c.y, ww.y, acc);
      acc = fmaf(a.z * c.z, ww.z, acc);
      acc = fmaf(a.w * c.w, ww.w, acc);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) pred[l] = acc + b[0];
  }
}

// per-position gradient rows: G[2l] = g*w*H[i1], G[2l+1] = g*w*H[i0]; Pm[l] = g*H[i0]*H[i1]  (g = dpred[l])
__global__ void __launch_bounds__(kRowThreads) k_readout_bwd_rows(const float* __restrict__ H, const int64_t* __restrict__ idx,
                                                                  int64_t sidx, int64_t L, int C, const float* __restrict__ w,
                                                                  const float* __restrict__ dpred, float* __restrict__ G,
                                                                  float* __restrict__ Pm) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ H4 = reinterpret_cast<const float4*>(H);
  const float4 ww = __ldg(reinterpret_cast<const float4*>(w) + rs.c4);
  float4* __restrict__ G4 = reinterpret_cast<float4*>(G);
  float4* __restrict__ P4 = reinterpret_cast<float4*>(Pm);
  for (int64_t l = (int64_t)blockIdx.x * rs.slots + rs.slot; l < L; l += (int64_t)gridDim.x * rs.slots) {
    const int64_t i0 = idx[(2 * l) * sidx], i1 = idx[(2 * l + 1) * sidx];
    const float g = dpred[l];
    const float4 a = ldg_cached(H4 + i0 * rs.cv + rs.c4), c = ldg_cached(H4 + i1 * rs.cv + rs.c4);
    const float4 gw = make_float4(g * ww.x, g * ww.y, g * ww.z, g * ww.w);
    G4[(2 * l) * rs.cv + rs.c4] = f4_mul(gw, c);
    G4[(2 * l + 1) * rs.cv + rs.c4] = f4_mul(gw, a);
    const float4 ac = f4_mul(a, c);
    P4[l * rs.cv + rs.c4] = make_float4(g * ac.x, g * ac.y, g * ac.z, g * ac.w);
  }
}

// dH[idx[j]] = sum of G[j'] over all positions j' with idx[j'] == idx[j], summed in position order.
// `order` = positions sorted by (idx value, position) (twowl_csr_build). One row slot per sorted position;
// the first position of each run of equal keys does the run.
__global__ void __launch_bounds__(kRowThreads) k_scatter_rows_sorted(const float* __restrict__ G, const int32_t* __restrict__ order,
                                                                     const int64_t* __restrict__ idx, int64_t sidx, int64_t n,
                                                                     int C, float* __restrict__ dH) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ G4 = reinterpret_cast<const float4*>(G);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(dH);
  for (int64_t j = (int64_t)blockIdx.x * rs.slots + rs.slot; j < n; j += (int64_t)gridDim.x * rs.slots) {
    const int64_t key = idx[(int64_t)order[j] * sidx];
    if (j > 0 && idx[(int64_t)order[j - 1] * sidx] == key) continue;
    float4 acc = f4_zero();
    for (int64_t q = j; q < n && idx[(int64_t)order[q] * sidx] == key; ++q) f4_add(acc, G4[(int64_t)order[q] * rs.cv + rs.c4]);
    o4[key * rs.cv + rs.c4] = acc;
  }
}

__global__ void k_sum_vec(const float* __restrict__ v, int64_t n, float* __restrict__ out) {
  // single CTA, fixed order: per-thread strided double partials, then a tree over 256 threads
  __shared__ double s[256];
  double a = 0;
  for (int64_t i = threadIdx.x; i < n; i += 256) a += (double)v[i];
  s[threadIdx.x] = a;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if ((int)threadIdx.x < d) s[threadIdx.x] += s[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)s[0];
}

// ---------------------------------------------------------------- structured wedge path ----------
__global__ void __launch_bounds__(kRowThreads) k_wedge_cnt_init(const int64_t* __restrict__ in_ptr, int64_t N, int32_t* __restrict__ cnt) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
    cnt[i] = (int32_t)(in_ptr[i + 1] - in_ptr[i]);
}
__global__ void __launch_bounds__(kRowThreads) k_wedge_cnt_block(const int32_t* __restrict__ dst_e, int64_t E, int64_t N,
                                                                 const uint8_t* __restrict__ blocked, int32_t* __restrict__ cnt) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < E; a += (int64_t)gridDim.x * blockDim.x) {
    const int32_t i = dst_e[a];
    if (blocked[a] && i >= 0 && i < N) atomicSub(&cnt[i], 1);  // integer atomics: order-independent result
  }
}
// rows [row_lo, row_hi) of the pair table -> entries [out_off, out_off + row_hi - row_lo) of the [2, Rout] outputs
// (the whole table: row_lo = 0, row_hi = Rout = R, out_off = 0; a rank's block of the row-sharded path is two ranges - its
// slice of the observed pairs, then its slice of the prediction pairs - written one after the other)
__global__ void __launch_bounds__(kRowThreads) k_wedge_rows(const int32_t* __restrict__ src, const int32_t* __restrict__ dst_e,
                                                            int64_t E, int64_t R, int64_t N, const uint8_t* __restrict__ blocked,
                                                            const int32_t* __restrict__ cnt, int64_t row_lo, int64_t row_hi,
                                                            int64_t Rout, int64_t out_off, int32_t* __restrict__ centre_,
                                                            float* __restrict__ dinv_, float* __restrict__ selfw_,
                                                            int32_t* __restrict__ bnode_) {
  // the outputs are addressed by the table's row id: [q * Rout + out_off + (b - row_lo)] = base[q * Rout + b]
  int32_t* const centre = centre_ + (out_off - row_lo);
  float* const dinv = dinv_ + (out_off - row_lo);
  float* const selfw = selfw_ + (out_off - row_lo);
  int32_t* const bnode = bnode_ + (out_off - row_lo);
  for (int64_t b = row_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < row_hi; b += (int64_t)gridDim.x * blockDim.x) {
    // direction 0 (edge2 = [a^1; b]): row b is fed by the in-list of src[b]; its id-self-loop is a = b^1
    // direction 1 (edge2_r = [a; b^1]): row b is fed by the in-list of src[b^1]; its id-self-loop is a = b
    const int64_t mate = b ^ 1;
    const int32_t c0 = src[b];
    const int32_t c1 = mate < R ? src[mate] : -1;
    const int n0 = (c0 >= 0 && c0 < N) ? cnt[c0] : 0;
    const int n1 = (c1 >= 0 && c1 < N) ? cnt[c1] : 0;
    const bool self0 = mate < E && n0 > 0 && dst_e[mate] == c0 && !(blocked && blocked[mate]);
    const bool self1 = b < E && n1 > 0 && dst_e[b] == c1 && !(blocked && blocked[b]);
    const float d0 = rsqrtf_exact((float)(n0 - (self0 ? 1 : 0) + 1));
    const float d1 = rsqrtf_exact((float)(n1 - (self1 ? 1 : 0) + 1));
    centre[b] = (c0 >= 0 && c0 < N) ? c0 : -1;
    centre[Rout + b] = (c1 >= 0 && c1 < N) ? c1 : -1;
    dinv[b] = d0;
    dinv[Rout + b] = d1;
    selfw[b] = self0 ? 0.f : d0 * d0;
    selfw[Rout + b] = self1 ? 0.f : d1 * d1;
    // backward: row b is a source of S_d[node] iff its feeding edge (b^1 for direction 0, b for direction 1) is live
    int32_t n0b = -1, n1b = -1;
    if (mate < E && !(blocked && blocked[mate])) {
      const int32_t nd = dst_e[mate];
      if (nd >= 0 && nd < N) n0b = nd;
    }
    if (b < E && !(blocked && blocked[b])) {
      const int32_t nd = dst_e[b];
      if (nd >= 0 && nd < N) n1b = nd;
    }
    bnode[b] = n0b;
    bnode[Rout + b] = n1b;
  }
}

// out[b] = dinv[b]*S[centre[b]] + selfw[b]*Z[b] + bias
__global__ void __launch_bounds__(kRowThreads) k_wedge_apply_fwd(const float* __restrict__ S, const float* __restrict__ Z,
                                                                 const int32_t* __restrict__ centre, const float* __restrict__ dinv,
                                                                 const float* __restrict__ selfw, const float* __restrict__ bias,
                                                                 int64_t R, int C, float* __restrict__ out) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ S4 = reinterpret_cast<const float4*>(S);
  const float4* __restrict__ Z4 = reinterpret_cast<const float4*>(Z);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(out);
  const float4 bb = bias ? __ldg(reinterpret_cast<const float4*>(bias) + rs.c4) : f4_zero();
  for (int64_t r = (int64_t)blockIdx.x * rs.slots + rs.slot; r < R; r += (int64_t)gridDim.x * rs.slots) {
    float4 o = bb;
    const int32_t c = centre[r];
    const float sw = selfw[r];
    if (c >= 0) f4_fma(o, dinv[r], ldg_cached(S4 + (int64_t)c * rs.cv + rs.c4));
    if (sw != 0.f) f4_fma(o, sw, ldg_stream(Z4 + r * rs.cv + rs.c4));
    stg_stream(o4 + r * rs.cv + rs.c4, o);
  }
}

// dZ[r] = selfw[r]*dO[r] + (row r is a source of S ? dinv[r]*dS[node] : 0)
// direction 0: S0[i] sums rows a^1 over unblocked a with dst_e[a] = i  ->  row r feeds via a = r^1
// direction 1: S1[i] sums rows a                                          ->  row r feeds via a = r
__global__ void __launch_bounds__(kRowThreads) k_wedge_apply_bwd(const float* __restrict__ dS, const float* __restrict__ dO,
                                                                 const int32_t* __restrict__ dst_e,
                                                                 const uint8_t* __restrict__ blocked, int64_t E, int64_t N,
                                                                 const float* __restrict__ dinv, const float* __restrict__ selfw,
                                                                 int direction, int64_t R, int C, float* __restrict__ dZ) {
  const RowSlots rs(C);
  if (rs.slot < 0) return;
  const float4* __restrict__ S4 = reinterpret_cast<const float4*>(dS);
  const float4* __restrict__ O4 = reinterpret_cast<const float4*>(dO);
  float4* __restrict__ z4 = reinterpret_cast<float4*>(dZ);
  for (int64_t r = (int64_t)blockIdx.x * rs.slots + rs.slot; r < R; r += (int64_t)gridDim.x * rs.slots) {
    float4 o = f4_zero();
    const float sw = selfw[r];
    if (sw != 0.f) f4_fma(o, sw, ldg_stream(O4 + r * rs.cv + rs.c4));
    const int64_t a = direction == 0 ? (r ^ 1) : r;
    if (a < E && !(blocked && blocked[a])) {
      const int32_t node = dst_e[a];
      if (node >= 0 && node < N) f4_fma(o, dinv[r], ldg_cached(S4 + (int64_t)node * rs.cv + rs.c4));
    }
    stg_stream(z4 + r * rs.cv + rs.c4, o);
  }
}

static int check_c(const char* op, int C) {
  TW_CHECK_ARG(C >= 4 && (C & 3) == 0 && C <= 1024, "%s: C=%d must be a multiple of 4 in [4,1024]", op, C);
  return 0;
}

}  // namespace twowl

using namespace twowl;

extern "C" int twowl_gather_rows(const float* W, int64_t rows_w, const int64_t* idx, int64_t stride, int64_t n, int32_t C,
                                 float* out, void* stream) {
  if (int rc = check_c("gather_rows", C)) return rc;
  TW_CHECK_ARG(aligned16(W) && aligned16(out), "gather_rows: W/out must be 16-byte aligned");
  if (n <= 0) return 0;
  k_gather_rows<<<row_grid(n, C), kRowThreads, 0, (cudaStream_t)stream>>>(W, rows_w, idx, stride, n, C, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_pair_init_fwd(const float* X, const int32_t* src, const int32_t* dst, int64_t R, int32_t C, int32_t pairs,
                                   float* out, void* stream) {
  if (int rc = check_c("pair_init_fwd", C)) return rc;
  TW_CHECK_ARG(aligned16(X) && aligned16(out), "pair_init_fwd: X/out must be 16-byte aligned");
  TW_CHECK_ARG(pairs == 0 || (pairs == 1 && R % 2 == 0), "pair_init_fwd: pairs = %d needs 0, or 1 with an even R", pairs);
  const int64_t rows = R >> pairs;
  if (rows <= 0) return 0;
  k_pair_init<<<row_grid(rows, C), kRowThreads, 0, (cudaStream_t)stream>>>(X, src, dst, rows, C, pairs, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_readout_fwd(const float* H, const int64_t* idx, int64_t sidx, int64_t L, int32_t C, const float* w,
                                 const float* b, float* pred, void* stream) {
  if (int rc = check_c("readout_fwd", C)) return rc;
  TW_CHECK_ARG(aligned16(H) && aligned16(w), "readout_fwd: H/w must be 16-byte aligned");
  if (L <= 0) return 0;
  k_readout_fwd<<<grid_for(L, kRowThreads / 32, 8), kRowThreads, 0, (cudaStream_t)stream>>>(H, idx, sidx, L, C, w, b, pred);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_colsum_workspace_bytes(int64_t M, int32_t C);
extern "C" int twowl_colsum(const float* x, int64_t M, int32_t C, float* out, void* ws, size_t ws_bytes, void* stream);

extern "C" size_t twowl_readout_bwd_workspace_bytes(int64_t L, int32_t C) {
  const size_t l = (size_t)(L > 0 ? L : 1);
  return align_up(2 * l * C * sizeof(float)) + align_up(l * C * sizeof(float)) + twowl_colsum_workspace_bytes(L, C);
}

extern "C" int twowl_readout_bwd(const float* H, const int64_t* idx, int64_t sidx, int64_t L, int32_t C, const float* w,
                                 const float* dpred, const int32_t* order, float* dH, float* dw, float* db, void* ws,
                                 size_t ws_bytes, void* stream) {
  if (int rc = check_c("readout_bwd", C)) return rc;
  TW_CHECK_ARG(aligned16(H) && aligned16(w) && aligned16(dH), "readout_bwd: H/w/dH must be 16-byte aligned");
  TW_CHECK_WS(ws_bytes, twowl_readout_bwd_workspace_bytes(L, C));
  cudaStream_t s = (cudaStream_t)stream;
  if (L <= 0) {
    TW_CUDA(cudaMemsetAsync(dw, 0, (size_t)C * sizeof(float), s));
    TW_CUDA(cudaMemsetAsync(db, 0, sizeof(float), s));
    return 0;
  }
  Carver c(ws);
  float* G = c.take<float>(2 * (size_t)L * C);
  float* Pm = c.take<float>((size_t)L * C);
  void* cs_ws = c.take<char>(twowl_colsum_workspace_bytes(L, C));
  k_readout_bwd_rows<<<row_grid(L, C), kRowThreads, 0, s>>>(H, idx, sidx, L, C, w, dpred, G, Pm);
  k_scatter_rows_sorted<<<row_grid(2 * L, C), kRowThreads, 0, s>>>(G, order, idx, sidx, 2 * L, C, dH);
  TW_LAUNCH_CHECK();
  if (int rc = twowl_colsum(Pm, L, C, dw, cs_ws, twowl_colsum_workspace_bytes(L, C), stream)) return rc;
  k_sum_vec<<<1, 256, 0, s>>>(dpred, L, db);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_wedge_prepare(const int32_t* src, const int32_t* dst_e, int64_t E, int64_t R, int64_t N,
                                   const uint8_t* blocked, const int64_t* in_ptr, int64_t lo0, int64_t hi0, int64_t lo1, int64_t hi1,
                                   int32_t* cnt, int32_t* centre, float* dinv, float* selfw, int32_t* bnode, void* stream) {
  TW_CHECK_ARG(E >= 0 && R >= E && N >= 0, "wedge_prepare: need 0 <= E <= R and N >= 0");
  TW_CHECK_ARG(lo0 >= 0 && lo0 <= hi0 && hi0 <= lo1 && lo1 <= hi1 && hi1 <= R && !((lo0 | hi0 | lo1 | hi1) & 1),
               "wedge_prepare: [%lld, %lld) and [%lld, %lld) must be even-bounded, ordered, disjoint ranges of the %lld pair rows",
               (long long)lo0, (long long)hi0, (long long)lo1, (long long)hi1, (long long)R);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n0 = hi0 - lo0, n1 = hi1 - lo1;
  if (N > 0) k_wedge_cnt_init<<<grid_for(N, kRowThreads), kRowThreads, 0, s>>>(in_ptr, N, cnt);
  if (blocked && E > 0 && N > 0) k_wedge_cnt_block<<<grid_for(E, kRowThreads), kRowThreads, 0, s>>>(dst_e, E, N, blocked, cnt);
  if (n0 > 0)
    k_wedge_rows<<<grid_for(n0, kRowThreads), kRowThreads, 0, s>>>(src, dst_e, E, R, N, blocked, cnt, lo0, hi0, n0 + n1, 0, centre, dinv,
                                                                   selfw, bnode);
  if (n1 > 0)
    k_wedge_rows<<<grid_for(n1, kRowThreads), kRowThreads, 0, s>>>(src, dst_e, E, R, N, blocked, cnt, lo1, hi1, n0 + n1, n0, centre, dinv,
                                                                   selfw, bnode);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_wedge_apply_fwd(const float* S, const float* Z, const int32_t* centre, const float* dinv,
                                     const float* selfw, const float* bias, int64_t R, int32_t C, float* out, void* stream) {
  if (int rc = check_c("wedge_apply_fwd", C)) return rc;
  TW_CHECK_ARG(aligned16(S) && aligned16(Z) && aligned16(out) && aligned16(bias), "wedge_apply_fwd: 16-byte alignment required");
  if (R <= 0) return 0;
  k_wedge_apply_fwd<<<row_grid(R, C), kRowThreads, 0, (cudaStream_t)stream>>>(S, Z, centre, dinv, selfw, bias, R, C, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_wedge_apply_bwd(const float* dS, const float* dO, const int32_t* dst_e, const uint8_t* blocked, int64_t E,
                                     int64_t N, const float* dinv, const float* selfw, int32_t direction, int64_t R, int32_t C,
                                     float* dZ, void* stream) {
  if (int rc = check_c("wedge_apply_bwd", C)) return rc;
  TW_CHECK_ARG(aligned16(dS) && aligned16(dO) && aligned16(dZ), "wedge_apply_bwd: 16-byte alignment required");
  TW_CHECK_ARG(direction == 0 || direction == 1, "wedge_apply_bwd: direction must be 0 or 1");
  if (R <= 0) return 0;
  k_wedge_apply_bwd<<<row_grid(R, C), kRowThreads, 0, (cudaStream_t)stream>>>(dS, dO, dst_e, blocked, E, N, dinv, selfw, direction,
                                                                            R, C, dZ);
  TW_LAUNCH_CHECK();
  return 0;
}
