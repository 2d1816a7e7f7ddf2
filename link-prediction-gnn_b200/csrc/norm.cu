// norm.cu - GraphNorm (PyG 2.3.1 semantics, batch=None) fused with the Dropout and ReLU that follow it in
// the reference's Seq block (TwoWL/model/model.py:36-41, :53-55), forward and backward, plus column sums.
//
// All kernels stream [M, C] fp32 row-major matrices with 128-bit accesses: thread t of a 256-thread CTA owns
// float4 column (t % cv) of row-slot (t / cv), cv = C/4, so a warp reads consecutive 16-byte words of
// consecutive rows (fully coalesced for every C % 4 == 0, including C = 24). Column reductions are
// two-level with a fixed order (per-thread fp32 partials over shifted values -> per-CTA double ->
// finalize in CTA order): deterministic, no atomics. HBM-bound: stats = 1 read, apply = 1 read + 1 write,
// bwd = 2 reads + (2 reads + 1 write).
#include "common.cuh"

namespace twowl {

constexpr int kNormThreads = 256;
// Readout row ids (twowl_gn2_readout_*): any negative id = "this link is masked" (a row-sharded caller masks the links outside
// its block); kMaskedTail additionally promises that EVERY later link of the list is masked as well (a caller that packed its
// own links at the front, twowl_b200.rowshard.own_links_first) - the kernels stop there instead of scanning the tail.
constexpr int64_t kMaskedTail = -2;
constexpr int kNormMaxCtas = kNumSMs * 4;

struct RowMap {
  int cv;        // float4 per row
  int slots;     // row slots per CTA iteration
  int slot;      // this thread's row slot (or -1 when idle)
  int c4;        // this thread's float4 column
  __device__ RowMap(int C) {
    cv = C >> 2;
    slots = kNormThreads / cv;
    const int t = threadIdx.x;
    slot = (t < slots * cv) ? t / cv : -1;
    c4 = t % cv;
  }
};

// Column sums without long fp32 chains: a thread's fp32 running sums are folded into double accumulators every kFoldRows rows
// (a grid-stride thread of a 1 M-row pass adds ~110 rows, of a 60 M-row pass ~6 000; as one fp32 chain that put ~1e-6 of
// relative error into GraphNorm's mean / variance and into every column-sum gradient - 5-13 x what torch's cascaded fp32 sums
// leave, measured stage by stage with tools/diag_node.py).
constexpr int kFoldRows = 8;
// The double accumulators live in shared memory, [value][component][thread] (conflict-free, no registers: in registers they
// cost k_gn2_readout_bwd_rows its second CTA per SM).
template <int NV>
struct ColFold {
  double* base;
  int n;
  __device__ __forceinline__ ColFold() : n(0) {
    extern __shared__ double s_fold[];
    base = s_fold + threadIdx.x;
#pragma unroll
    for (int i = 0; i < NV * 4; ++i) base[i * kNormThreads] = 0.0;
  }
  __device__ __forceinline__ void flush(float4 (&val)[NV]) {
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      double* o = base + (v * 4) * kNormThreads;
      o[0] += (double)val[v].x, o[kNormThreads] += (double)val[v].y;
      o[2 * kNormThreads] += (double)val[v].z, o[3 * kNormThreads] += (double)val[v].w;
      val[v] = f4_zero();
    }
    n = 0;
  }
  __device__ __forceinline__ void tick(float4 (&val)[NV]) {
    if (++n == kFoldRows) flush(val);
  }
};

// The CTA's row slots added in slot order: part[blockIdx.x][v][C] (thread slot * cv + c4 holds columns 4 c4 .. 4 c4 + 3).
template <int NV>
__device__ __forceinline__ void cta_col_reduce_d(const RowMap& rm, const ColFold<NV>&, double* __restrict__ part, int C) {
  extern __shared__ double s_fold[];
  __syncthreads();
  for (int i = threadIdx.x; i < NV * C; i += kNormThreads) {
    const int v = i / C, c = i % C;
    const double* col = s_fold + (size_t)(v * 4 + (c & 3)) * kNormThreads + (c >> 2);
    double a = 0;
    for (int sl = 0; sl < rm.slots; ++sl) a += col[sl * rm.cv];
    part[((size_t)blockIdx.x * NV + v) * C + c] = a;
  }
}

// ---------------------------------------------------------------- forward statistics -------------
__global__ void __launch_bounds__(kNormThreads) k_gn_stats_partial(const float* __restrict__ x, int64_t M, int C,
                                                                   double* __restrict__ part) {
  const RowMap rm(C);
  float4 v[2] = {f4_zero(), f4_zero()};
  ColFold<2> fold;
  if (rm.slot >= 0) {
    const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
    const float4 sh = __ldg(x4 + rm.c4);  // shift = first row: keeps the squared sums well conditioned
    for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
      float4 a = ldg_stream(x4 + r * rm.cv + rm.c4);
      a.x -= sh.x, a.y -= sh.y, a.z -= sh.z, a.w -= sh.w;
      f4_add(v[0], a);
      v[1].x = fmaf(a.x, a.x, v[1].x), v[1].y = fmaf(a.y, a.y, v[1].y);
      v[1].z = fmaf(a.z, a.z, v[1].z), v[1].w = fmaf(a.w, a.w, v[1].w);
      fold.tick(v);
    }
    fold.flush(v);
  }
  cta_col_reduce_d<2>(rm, fold, part, C);
}

__global__ void k_gn_stats_final(const double* __restrict__ part, int nparts, const float* __restrict__ x, int64_t M, int C,
                                 const float* __restrict__ mean_scale, float eps, float* __restrict__ stats) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s = 0, q = 0;
  for (int b = 0; b < nparts; ++b) {
    s += part[((size_t)b * 2 + 0) * C + c];
    q += part[((size_t)b * 2 + 1) * C + c];
  }
  const double sh = (double)x[c];
  const double ms = s / (double)M;                 // mean of shifted values
  const double mean = sh + ms;
  double var = q / (double)M - ms * ms;            // Var(x)
  if (var < 0) var = 0;
  const double a = (double)mean_scale[c];
  const double var_shifted = var + (1.0 - a) * (1.0 - a) * mean * mean;  // E[(x - a*mean)^2]
  stats[c] = (float)mean;
  stats[C + c] = (float)(1.0 / sqrt(var_shifted + (double)eps));
}

// ---------------------------------------------------------------- forward apply ------------------
__global__ void __launch_bounds__(kNormThreads) k_gn_apply(const float* __restrict__ x, int64_t M, int C,
                                                           const float* __restrict__ stats, const float* __restrict__ weight,
                                                           const float* __restrict__ bias, const float* __restrict__ mean_scale,
                                                           uint32_t thresh, float inv_keep, uint64_t seed, int relu,
                                                           const float* addend, float* out) {
  seed = resolve_seed(seed);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  if (rm.slot < 0) return;
  const int c0 = rm.c4 * 4;
  float sc[4], of[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    sc[i] = weight[c0 + i] * stats[C + c0 + i];
    of[i] = bias[c0 + i] - sc[i] * mean_scale[c0 + i] * stats[c0 + i];
  }
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
  float4* o4 = reinterpret_cast<float4*>(out);
  const float4* a4 = reinterpret_cast<const float4*>(addend);
  for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
    const int64_t e = r * rm.cv + rm.c4;
    const float4 a = ldg_stream(x4 + e);
    float y[4] = {fmaf(sc[0], a.x, of[0]), fmaf(sc[1], a.y, of[1]), fmaf(sc[2], a.z, of[2]), fmaf(sc[3], a.w, of[3])};
    if (thresh) {
#pragma unroll
      for (int i = 0; i < 4; ++i) y[i] *= drop_scale(seed, (uint64_t)e * 4 + i, thresh, inv_keep);
    }
    if (relu) {
#pragma unroll
      for (int i = 0; i < 4; ++i) y[i] = fmaxf(y[i], 0.f);
    }
    float4 o = make_float4(y[0], y[1], y[2], y[3]);
    if (a4) f4_add(o, a4[e]);
    o4[e] = o;
  }
}

// ---------------------------------------------------------------- backward -----------------------
// g_y = dout * dropout_scale * [relu: y_dropped > 0];  n = (x - a*mean)*inv
__device__ __forceinline__ void gn_gy(const float4& a, const float4& d, const float (&sc)[4], const float (&of)[4],
                                      const float (&nm)[4], const float (&ni)[4], uint32_t thresh, float inv_keep,
                                      uint64_t seed, uint64_t e, int relu, float (&gy)[4], float (&n)[4]) {
  const float xa[4] = {a.x, a.y, a.z, a.w};
  const float da[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    n[i] = (xa[i] - nm[i]) * ni[i];
    float g = da[i];
    float keep = 1.f;
    if (thresh) keep = drop_scale(seed, e * 4 + i, thresh, inv_keep);
    g *= keep;
    if (relu) {
      const float y = fmaf(sc[i], xa[i], of[i]) * keep;
      if (!(y > 0.f)) g = 0.f;
    }
    gy[i] = g;
  }
}

struct GnCols {
  float sc[4], of[4], nm[4], ni[4];
  __device__ GnCols(int C, int c0, const float* stats, const float* weight, const float* bias, const float* mean_scale) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ni[i] = stats[C + c0 + i];
      nm[i] = mean_scale[c0 + i] * stats[c0 + i];
      sc[i] = weight[c0 + i] * ni[i];
      of[i] = bias[c0 + i] - sc[i] * nm[i];
    }
  }
};

__global__ void __launch_bounds__(kNormThreads) k_gn_bwd_partial(const float* __restrict__ x, const float* __restrict__ dout,
                                                                 int64_t M, int C, const float* __restrict__ stats,
                                                                 const float* __restrict__ weight, const float* __restrict__ bias,
                                                                 const float* __restrict__ mean_scale, uint32_t thresh,
                                                                 float inv_keep, uint64_t seed, int relu,
                                                                 double* __restrict__ part) {
  seed = resolve_seed(seed);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  float4 v[2] = {f4_zero(), f4_zero()};
  ColFold<2> fold;
  if (rm.slot >= 0) {
    const GnCols cc(C, rm.c4 * 4, stats, weight, bias, mean_scale);
    const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
    const float4* __restrict__ d4 = reinterpret_cast<const float4*>(dout);
    for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
      const int64_t e = r * rm.cv + rm.c4;
      float gy[4], n[4];
      gn_gy(ldg_cached(x4 + e), ldg_cached(d4 + e), cc.sc, cc.of, cc.nm, cc.ni, thresh, inv_keep, seed, (uint64_t)e, relu, gy, n);
      v[0].x += gy[0], v[0].y += gy[1], v[0].z += gy[2], v[0].w += gy[3];
      v[1].x = fmaf(gy[0], n[0], v[1].x), v[1].y = fmaf(gy[1], n[1], v[1].y);
      v[1].z = fmaf(gy[2], n[2], v[1].z), v[1].w = fmaf(gy[3], n[3], v[1].w);
      fold.tick(v);
    }
    fold.flush(v);
  }
  cta_col_reduce_d<2>(rm, fold, part, C);
}

// sums[0:C] = A = sum g_y, sums[C:2C] = B = sum g_y*n, sums[2C:3C] = (alpha/M) * sum g_o   (fp32, for pass 2)
// dparams[0:C] = dweight = B, [C:2C] = dbias = A, [2C:3C] = dmean_scale = -mean * sum g_o, [3C:4C] = colsum(dx)
// one WARP per column: lane l adds the CTA partials l, l+32, ... then a fixed-order xor tree (deterministic)
__device__ __forceinline__ double warp_part_sum(const double* __restrict__ part, int nparts, int nv, int v, int C, int c) {
  const int lane = threadIdx.x & 31;
  double a = 0;
  for (int b = lane; b < nparts; b += 32) a += part[((size_t)b * nv + v) * C + c];
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
  return a;
}

__global__ void k_gn_bwd_final(const double* __restrict__ part, int nparts, int nv, int voff, int64_t M, int C,
                               const float* __restrict__ stats, const float* __restrict__ weight,
                               const float* __restrict__ mean_scale, float* __restrict__ sums, float* __restrict__ dparams) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= C) return;
  const double A = warp_part_sum(part, nparts, nv, voff + 0, C, c);
  const double B = warp_part_sum(part, nparts, nv, voff + 1, C, c);
  if ((threadIdx.x & 31) != 0) return;
  const double mean = stats[c], inv = stats[C + c], w = weight[c], a = mean_scale[c];
  // sum_rows n = inv * M * mean * (1 - a);  sum g_o = inv*w*(A - (B/M) * sum n)
  const double sum_go = inv * w * (A - B * inv * mean * (1.0 - a));
  sums[c] = (float)A;
  sums[C + c] = (float)(B / (double)M);
  sums[2 * C + c] = (float)(a * sum_go / (double)M);
  dparams[c] = (float)B;
  dparams[C + c] = (float)A;
  dparams[2 * C + c] = (float)(-mean * sum_go);
  dparams[3 * C + c] = (float)((1.0 - a) * sum_go);  // sum over rows of dx = sum g_o - a * sum g_o
}

__global__ void __launch_bounds__(kNormThreads) k_gn_bwd_dx(const float* __restrict__ x, const float* __restrict__ dout, int64_t M,
                                                            int C, const float* __restrict__ stats, const float* __restrict__ weight,
                                                            const float* __restrict__ bias, const float* __restrict__ mean_scale,
                                                            uint32_t thresh, float inv_keep, uint64_t seed, int relu,
                                                            const float* __restrict__ sums, float* __restrict__ dx) {
  seed = resolve_seed(seed);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  if (rm.slot < 0) return;
  const int c0 = rm.c4 * 4;
  const GnCols cc(C, c0, stats, weight, bias, mean_scale);
  float bm[4], corr[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    bm[i] = sums[C + c0 + i];
    corr[i] = sums[2 * C + c0 + i];
  }
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
  const float4* __restrict__ d4 = reinterpret_cast<const float4*>(dout);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(dx);
  for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
    const int64_t e = r * rm.cv + rm.c4;
    float gy[4], n[4], o[4];
    gn_gy(ldg_stream(x4 + e), ldg_stream(d4 + e), cc.sc, cc.of, cc.nm, cc.ni, thresh, inv_keep, seed, (uint64_t)e, relu, gy, n);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = cc.sc[i] * (gy[i] - n[i] * bm[i]) - corr[i];
    o4[e] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------- two branches sharing dout ------
// out = act(drop(GN_f(xf))) + act(drop(GN_r(xr)))  - the conv2s[i](x) + conv2s_r[i](x) sum of model.py:77 in one pass
__global__ void __launch_bounds__(kNormThreads) k_gn_apply2(const float* __restrict__ xf, const float* __restrict__ xr, int64_t M,
                                                            int C, const float* __restrict__ stf, const float* __restrict__ str_,
                                                            const float* __restrict__ wf, const float* __restrict__ bf,
                                                            const float* __restrict__ mf, const float* __restrict__ wr,
                                                            const float* __restrict__ br, const float* __restrict__ mr,
                                                            uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                            int relu, float* __restrict__ out) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  if (rm.slot < 0) return;
  const int c0 = rm.c4 * 4;
  const GnCols cf(C, c0, stf, wf, bf, mf), cr(C, c0, str_, wr, br, mr);
  const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
  const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
  float4* __restrict__ o4 = reinterpret_cast<float4*>(out);
  for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
    const int64_t e = r * rm.cv + rm.c4;
    const float4 a = ldg_stream(xf4 + e), b = ldg_stream(xr4 + e);
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float yf = fmaf(cf.sc[i], av[i], cf.of[i]), yr = fmaf(cr.sc[i], bv[i], cr.of[i]);
      if (thresh) {
        yf *= drop_scale(seed_f, (uint64_t)e * 4 + i, thresh, inv_keep);
        yr *= drop_scale(seed_r, (uint64_t)e * 4 + i, thresh, inv_keep);
      }
      if (relu) yf = fmaxf(yf, 0.f), yr = fmaxf(yr, 0.f);
      o[i] = yf + yr;
    }
    o4[e] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

__global__ void __launch_bounds__(kNormThreads) k_gn_bwd2_partial(const float* __restrict__ xf, const float* __restrict__ xr,
                                                                  const float* __restrict__ dout, int64_t M, int C,
                                                                  const float* __restrict__ stf, const float* __restrict__ str_,
                                                                  const float* __restrict__ wf, const float* __restrict__ bf,
                                                                  const float* __restrict__ mf, const float* __restrict__ wr,
                                                                  const float* __restrict__ br, const float* __restrict__ mr,
                                                                  uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                                  int relu, double* __restrict__ part) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  float4 v[4] = {f4_zero(), f4_zero(), f4_zero(), f4_zero()};
  ColFold<4> fold;
  if (rm.slot >= 0) {
    const int c0 = rm.c4 * 4;
    const GnCols cf(C, c0, stf, wf, bf, mf), cr(C, c0, str_, wr, br, mr);
    const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
    const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
    const float4* __restrict__ d4 = reinterpret_cast<const float4*>(dout);
    for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
      const int64_t e = r * rm.cv + rm.c4;
      const float4 d = ldg_cached(d4 + e);
      float gy[4], n[4];
      gn_gy(ldg_cached(xf4 + e), d, cf.sc, cf.of, cf.nm, cf.ni, thresh, inv_keep, seed_f, (uint64_t)e, relu, gy, n);
      v[0].x += gy[0], v[0].y += gy[1], v[0].z += gy[2], v[0].w += gy[3];
      v[1].x = fmaf(gy[0], n[0], v[1].x), v[1].y = fmaf(gy[1], n[1], v[1].y);
      v[1].z = fmaf(gy[2], n[2], v[1].z), v[1].w = fmaf(gy[3], n[3], v[1].w);
      gn_gy(ldg_cached(xr4 + e), d, cr.sc, cr.of, cr.nm, cr.ni, thresh, inv_keep, seed_r, (uint64_t)e, relu, gy, n);
      v[2].x += gy[0], v[2].y += gy[1], v[2].z += gy[2], v[2].w += gy[3];
      v[3].x = fmaf(gy[0], n[0], v[3].x), v[3].y = fmaf(gy[1], n[1], v[3].y);
      v[3].z = fmaf(gy[2], n[2], v[3].z), v[3].w = fmaf(gy[3], n[3], v[3].w);
      fold.tick(v);
    }
    fold.flush(v);
  }
  cta_col_reduce_d<4>(rm, fold, part, C);
}

__global__ void __launch_bounds__(kNormThreads) k_gn_bwd2_dx(const float* __restrict__ xf, const float* __restrict__ xr,
                                                             const float* __restrict__ dout, int64_t M, int C,
                                                             const float* __restrict__ stf, const float* __restrict__ str_,
                                                             const float* __restrict__ wf, const float* __restrict__ bf,
                                                             const float* __restrict__ mf, const float* __restrict__ wr,
                                                             const float* __restrict__ br, const float* __restrict__ mr,
                                                             uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                             int relu, const float* __restrict__ sums_f,
                                                             const float* __restrict__ sums_r, float* __restrict__ dxf,
                                                             float* __restrict__ dxr) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  if (rm.slot < 0) return;
  const int c0 = rm.c4 * 4;
  const GnCols cf(C, c0, stf, wf, bf, mf), cr(C, c0, str_, wr, br, mr);
  float bmf[4], cof[4], bmr[4], cor[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    bmf[i] = sums_f[C + c0 + i], cof[i] = sums_f[2 * C + c0 + i];
    bmr[i] = sums_r[C + c0 + i], cor[i] = sums_r[2 * C + c0 + i];
  }
  const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
  const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
  const float4* __restrict__ d4 = reinterpret_cast<const float4*>(dout);
  float4* __restrict__ of4 = reinterpret_cast<float4*>(dxf);
  float4* __restrict__ or4 = reinterpret_cast<float4*>(dxr);
  for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
    const int64_t e = r * rm.cv + rm.c4;
    const float4 d = ldg_stream(d4 + e), a = ldg_stream(xf4 + e), b = ldg_stream(xr4 + e);
    float gy[4], n[4], o[4];
    gn_gy(a, d, cf.sc, cf.of, cf.nm, cf.ni, thresh, inv_keep, seed_f, (uint64_t)e, relu, gy, n);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = cf.sc[i] * (gy[i] - n[i] * bmf[i]) - cof[i];
    of4[e] = make_float4(o[0], o[1], o[2], o[3]);
    gn_gy(b, d, cr.sc, cr.of, cr.nm, cr.ni, thresh, inv_keep, seed_r, (uint64_t)e, relu, gy, n);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = cr.sc[i] * (gy[i] - n[i] * bmr[i]) - cor[i];
    or4[e] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------- last pair layer + readout -------
// When a pair layer's output only feeds the readout x[idx] (model.py:77-83, the LAST conv2s/conv2s_r layer), the two
// GraphNorm(+Dropout+ReLU) branches are evaluated at the 2L selected rows only, and the backward exploits that the
// incoming gradient is zero outside those rows: column reductions over 2L positions, one dense pass for dxf / dxr.
__device__ __forceinline__ float4 gn2_row(const float4& a, const float4& b, const GnCols& cf, const GnCols& cr, uint32_t thresh,
                                          float inv_keep, uint64_t seed_f, uint64_t seed_r, int relu, uint64_t e) {
  const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
  float o[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float yf = fmaf(cf.sc[i], av[i], cf.of[i]), yr = fmaf(cr.sc[i], bv[i], cr.of[i]);
    if (thresh) {
      yf *= drop_scale(seed_f, e * 4 + i, thresh, inv_keep);
      yr *= drop_scale(seed_r, e * 4 + i, thresh, inv_keep);
    }
    if (relu) yf = fmaxf(yf, 0.f), yr = fmaxf(yr, 0.f);
    o[i] = yf + yr;
  }
  return make_float4(o[0], o[1], o[2], o[3]);
}

// pred[l] = sum_c hn[i0,c]*hn[i1,c]*w[c] + b. A lane GROUP of GW = 8 / 16 / 32 lanes (the smallest power of two >= C/4) owns a
// link, so a warp works on 32/GW links at once; two links per group are in flight per iteration (the row loads of a link depend
// on its idx load: one link at a time left this kernel latency-bound at 1.7 TB/s). Per-column constants are loaded once per
// thread. Fixed xor-shuffle tree inside the group: deterministic. C > 128 takes the strided loop of the general kernel.
template <int GW>
__global__ void __launch_bounds__(kNormThreads) k_gn2_readout_fwd_g(const float* __restrict__ xf, const float* __restrict__ xr, int C,
                                                                    const float* __restrict__ stf, const float* __restrict__ str_,
                                                                    const float* __restrict__ wf, const float* __restrict__ bf,
                                                                    const float* __restrict__ mf, const float* __restrict__ wr,
                                                                    const float* __restrict__ br, const float* __restrict__ mr,
                                                                    uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                                    int relu, const int64_t* __restrict__ idx, int64_t sidx, int64_t L,
                                                                    const float* __restrict__ w, const float* __restrict__ b,
                                                                    float* __restrict__ pred) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  constexpr int kPer = 32 / GW;
  const int lane = threadIdx.x & 31, sub = lane / GW, c4 = lane % GW;
  const int cv = C >> 2;
  const bool act = c4 < cv;
  const int cc = act ? c4 : 0;
  const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
  const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
  const GnCols cf(C, cc * 4, stf, wf, bf, mf), cr(C, cc * 4, str_, wr, br, mr);
  const float4 ww = act ? __ldg(reinterpret_cast<const float4*>(w) + cc) : f4_zero();
  const float bias = b[0];
  // groups of one warp leave the loop at different iterations: shuffles name only the group's own lanes
  const uint32_t gmask = GW == 32 ? 0xffffffffu : (((1u << (GW & 31)) - 1u) << (sub * GW));
  const int64_t grp0 = (((int64_t)blockIdx.x * kNormThreads + threadIdx.x) >> 5) * kPer + sub;
  const int64_t ngrp = (((int64_t)gridDim.x * kNormThreads) >> 5) * kPer;
  for (int64_t l0 = grp0; l0 < L; l0 += 2 * ngrp) {
    const int64_t l1 = l0 + ngrp;
    const bool two = l1 < L;
    // a negative row id = "this link is not mine" (a row-sharded caller masks the links outside its block): its logit is 0
    // and nothing is gathered for it (the loads below then read row 0)
    int64_t a0 = idx[(2 * l0) * sidx], a1 = idx[(2 * l0 + 1) * sidx];
    int64_t b0 = two ? idx[(2 * l1) * sidx] : a0, b1 = two ? idx[(2 * l1 + 1) * sidx] : a1;
    const bool va = a0 >= 0 && a1 >= 0, vb = b0 >= 0 && b1 >= 0;
    if (!va && !vb) {   // uniform over the lane group (its lanes share the two links): nothing to gather, nothing to reduce
      if (a0 == kMaskedTail) break;   // packed list: every later link is masked too (their logits were zeroed by the launcher)
      if (c4 == 0) {
        pred[l0] = 0.f;
        if (two) pred[l1] = 0.f;
      }
      continue;
    }
    if (!va) a0 = a1 = 0;
    if (!vb) b0 = b1 = 0;
    const int64_t ea0 = a0 * cv + cc, ea1 = a1 * cv + cc, eb0 = b0 * cv + cc, eb1 = b1 * cv + cc;
    const float4 fa0 = ldg_cached(xf4 + ea0), ra0 = ldg_cached(xr4 + ea0), fa1 = ldg_cached(xf4 + ea1), ra1 = ldg_cached(xr4 + ea1);
    const float4 fb0 = ldg_cached(xf4 + eb0), rb0 = ldg_cached(xr4 + eb0), fb1 = ldg_cached(xf4 + eb1), rb1 = ldg_cached(xr4 + eb1);
    const float4 ha0 = gn2_row(fa0, ra0, cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)ea0);
    const float4 ha1 = gn2_row(fa1, ra1, cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)ea1);
    const float4 hb0 = gn2_row(fb0, rb0, cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)eb0);
    const float4 hb1 = gn2_row(fb1, rb1, cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)eb1);
    float acc0 = 0.f, acc1 = 0.f;
    acc0 = fmaf(ha0.x * ha1.x, ww.x, acc0), acc0 = fmaf(ha0.y * ha1.y, ww.y, acc0);
    acc0 = fmaf(ha0.z * ha1.z, ww.z, acc0), acc0 = fmaf(ha0.w * ha1.w, ww.w, acc0);
    acc1 = fmaf(hb0.x * hb1.x, ww.x, acc1), acc1 = fmaf(hb0.y * hb1.y, ww.y, acc1);
    acc1 = fmaf(hb0.z * hb1.z, ww.z, acc1), acc1 = fmaf(hb0.w * hb1.w, ww.w, acc1);
    if (!act) acc0 = 0.f, acc1 = 0.f;
#pragma unroll
    for (int d = GW / 2; d > 0; d >>= 1) {
      acc0 += __shfl_xor_sync(gmask, acc0, d);
      acc1 += __shfl_xor_sync(gmask, acc1, d);
    }
    if (c4 == 0) {
      pred[l0] = va ? acc0 + bias : 0.f;
      if (two) pred[l1] = vb ? acc1 + bias : 0.f;
    }
  }
}

// general widths (C > 128): one warp per target link, columns strided over the lanes
__global__ void __launch_bounds__(kNormThreads) k_gn2_readout_fwd(const float* __restrict__ xf, const float* __restrict__ xr, int C,
                                                                  const float* __restrict__ stf, const float* __restrict__ str_,
                                                                  const float* __restrict__ wf, const float* __restrict__ bf,
                                                                  const float* __restrict__ mf, const float* __restrict__ wr,
                                                                  const float* __restrict__ br, const float* __restrict__ mr,
                                                                  uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                                  int relu, const int64_t* __restrict__ idx, int64_t sidx, int64_t L,
                                                                  const float* __restrict__ w, const float* __restrict__ b,
                                                                  float* __restrict__ pred) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const int lane = threadIdx.x & 31;
  const int cv = C >> 2;
  const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
  const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
  const float4* __restrict__ w4 = reinterpret_cast<const float4*>(w);
  const int64_t warp0 = ((int64_t)blockIdx.x * kNormThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kNormThreads) >> 5;
  for (int64_t l = warp0; l < L; l += nwarps) {
    const int64_t i0 = idx[(2 * l) * sidx], i1 = idx[(2 * l + 1) * sidx];
    if (i0 < 0 || i1 < 0) {   // not this rank's link (see k_gn2_readout_fwd_g); warp-uniform
      if (i0 == kMaskedTail) break;
      if (lane == 0) pred[l] = 0.f;
      continue;
    }
    float acc = 0.f;
    for (int c4 = lane; c4 < cv; c4 += 32) {
      const GnCols cf(C, c4 * 4, stf, wf, bf, mf), cr(C, c4 * 4, str_, wr, br, mr);
      const int64_t e0 = i0 * cv + c4, e1 = i1 * cv + c4;
      const float4 h0 = gn2_row(ldg_cached(xf4 + e0), ldg_cached(xr4 + e0), cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)e0);
      const float4 h1 = gn2_row(ldg_cached(xf4 + e1), ldg_cached(xr4 + e1), cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)e1);
      const float4 ww = __ldg(w4 + c4);
      acc = fmaf(h0.x * h1.x, ww.x, acc);
      acc = fmaf(h0.y * h1.y, ww.y, acc);
      acc = fmaf(h0.z * h1.z, ww.z, acc);
      acc = fmaf(h0.w * h1.w, ww.w, acc);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) pred[l] = acc + b[0];
  }
}

// per selected position j (row a = idx[j], partner row b = idx[j^1], link l = j/2):
//   G[j] = dpred[l] * w * hn[b]   (gradient w.r.t. hn[a]),  and the column partial sums of both GraphNorm backwards
//   (sum g_y, sum g_y*n per branch) plus dw = sum_l dpred[l] * hn[a]*hn[b] and db = sum_l dpred[l] (even positions only).
__global__ void __launch_bounds__(kNormThreads) k_gn2_readout_bwd_rows(const float* __restrict__ xf, const float* __restrict__ xr, int C,
                                                                       const float* __restrict__ stf, const float* __restrict__ str_,
                                                                       const float* __restrict__ wf, const float* __restrict__ bf,
                                                                       const float* __restrict__ mf, const float* __restrict__ wr,
                                                                       const float* __restrict__ br, const float* __restrict__ mr,
                                                                       uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                                       int relu, const int64_t* __restrict__ idx, int64_t sidx, int64_t L,
                                                                       const float* __restrict__ w, const float* __restrict__ dpred,
                                                                       float* __restrict__ G, double* __restrict__ part) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  float4 v[6] = {f4_zero(), f4_zero(), f4_zero(), f4_zero(), f4_zero(), f4_zero()};
  ColFold<6> fold;
  if (rm.slot >= 0) {
    const int c0 = rm.c4 * 4;
    const GnCols cf(C, c0, stf, wf, bf, mf), cr(C, c0, str_, wr, br, mr);
    const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
    const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
    const float4 ww = __ldg(reinterpret_cast<const float4*>(w) + rm.c4);
    float4* __restrict__ G4 = reinterpret_cast<float4*>(G);
    for (int64_t j = (int64_t)blockIdx.x * rm.slots + rm.slot; j < 2 * L; j += (int64_t)gridDim.x * rm.slots) {
      const int64_t ra = idx[j * sidx], rb = idx[(j ^ 1) * sidx];
      if (ra == kMaskedTail) break;     // packed list: every later position is masked too
      if (ra < 0 || rb < 0) continue;   // not this rank's link: no contribution to the column sums; its G row is never read
                                        // (the row chains hold valid positions only), so it is not written either
      const float g = dpred[j >> 1];
      const int64_t ea = ra * rm.cv + rm.c4, eb = rb * rm.cv + rm.c4;
      const float4 af = ldg_cached(xf4 + ea), ar = ldg_cached(xr4 + ea);
      const float4 hb = gn2_row(ldg_cached(xf4 + eb), ldg_cached(xr4 + eb), cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)eb);
      const float4 d = make_float4(g * ww.x * hb.x, g * ww.y * hb.y, g * ww.z * hb.z, g * ww.w * hb.w);
      G4[j * rm.cv + rm.c4] = d;
      float gy[4], n[4];
      gn_gy(af, d, cf.sc, cf.of, cf.nm, cf.ni, thresh, inv_keep, seed_f, (uint64_t)ea, relu, gy, n);
      v[0].x += gy[0], v[0].y += gy[1], v[0].z += gy[2], v[0].w += gy[3];
      v[1].x = fmaf(gy[0], n[0], v[1].x), v[1].y = fmaf(gy[1], n[1], v[1].y);
      v[1].z = fmaf(gy[2], n[2], v[1].z), v[1].w = fmaf(gy[3], n[3], v[1].w);
      gn_gy(ar, d, cr.sc, cr.of, cr.nm, cr.ni, thresh, inv_keep, seed_r, (uint64_t)ea, relu, gy, n);
      v[2].x += gy[0], v[2].y += gy[1], v[2].z += gy[2], v[2].w += gy[3];
      v[3].x = fmaf(gy[0], n[0], v[3].x), v[3].y = fmaf(gy[1], n[1], v[3].y);
      v[3].z = fmaf(gy[2], n[2], v[3].z), v[3].w = fmaf(gy[3], n[3], v[3].w);
      if ((j & 1) == 0) {
        const float4 ha = gn2_row(af, ar, cf, cr, thresh, inv_keep, seed_f, seed_r, relu, (uint64_t)ea);
        v[4].x = fmaf(g, ha.x * hb.x, v[4].x), v[4].y = fmaf(g, ha.y * hb.y, v[4].y);
        v[4].z = fmaf(g, ha.z * hb.z, v[4].z), v[4].w = fmaf(g, ha.w * hb.w, v[4].w);
        if (rm.c4 == 0) v[5].x += g;   // db = sum_l dpred[l], carried in column 0 of a sixth partial
      }
      fold.tick(v);
    }
    fold.flush(v);
  }
  cta_col_reduce_d<6>(rm, fold, part, C);
}

// per-row chains of the positions that select it: head[row] -> position -> next[position] -> ... -> -1.
// The chain ORDER is a race outcome and never reaches a result: consumers add a row's positions in ascending order.
// A position joins a chain only if its link is live, i.e. its partner id is not negative either: k_gn2_readout_bwd_rows writes
// no G row for a masked link, so a chain through one would add uninitialised workspace to the row's gradient.
__global__ void __launch_bounds__(kNormThreads) k_row_chains(const int64_t* __restrict__ idx, int64_t sidx, int64_t n, int64_t M,
                                                             int32_t* __restrict__ head, int32_t* __restrict__ next) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx[j * sidx];
    if (r == kMaskedTail) break;   // packed list: no later position selects a row, and next[] is only read along the chains
    const bool live = r >= 0 && r < M && idx[(j ^ 1) * sidx] >= 0;
    next[j] = live ? atomicExch(&head[r], (int32_t)j) : -1;
  }
}

__global__ void __launch_bounds__(kNormThreads, 3) k_gn_bwd2_dx_rows(const float* __restrict__ xf, const float* __restrict__ xr,
                                                                  const float* __restrict__ G, const int32_t* __restrict__ head,
                                                                  const int32_t* __restrict__ next, int64_t M, int C,
                                                                  const float* __restrict__ stf, const float* __restrict__ str_,
                                                                  const float* __restrict__ wf, const float* __restrict__ bf,
                                                                  const float* __restrict__ mf, const float* __restrict__ wr,
                                                                  const float* __restrict__ br, const float* __restrict__ mr,
                                                                  uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r,
                                                                  int relu, const float* __restrict__ sums_f,
                                                                  const float* __restrict__ sums_r, float* __restrict__ dxf,
                                                                  float* __restrict__ dxr) {
  seed_f = resolve_seed(seed_f); seed_r = resolve_seed(seed_r);   // a tagged seed is an address (common.cuh)
  const RowMap rm(C);
  if (rm.slot < 0) return;
  const int c0 = rm.c4 * 4;
  const GnCols cf(C, c0, stf, wf, bf, mf), cr(C, c0, str_, wr, br, mr);
  float bmf[4], cof[4], bmr[4], cor[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    bmf[i] = sums_f[C + c0 + i], cof[i] = sums_f[2 * C + c0 + i];
    bmr[i] = sums_r[C + c0 + i], cor[i] = sums_r[2 * C + c0 + i];
  }
  const float4* __restrict__ xf4 = reinterpret_cast<const float4*>(xf);
  const float4* __restrict__ xr4 = reinterpret_cast<const float4*>(xr);
  const float4* __restrict__ G4 = reinterpret_cast<const float4*>(G);
  float4* __restrict__ of4 = reinterpret_cast<float4*>(dxf);
  float4* __restrict__ or4 = reinterpret_cast<float4*>(dxr);
  auto chain_grad = [&](int64_t r) -> float4 {
    float4 d = f4_zero();
    const int h = __ldg(head + r);
    if (h >= 0) {
      if (__ldg(next + h) < 0) {
        d = ldg_cached(G4 + (int64_t)h * rm.cv + rm.c4);
      } else {  // the row is selected more than once: add its positions in ascending order
        int last = -1;
        for (;;) {
          int best = 0x7fffffff;
          for (int q = h; q >= 0; q = __ldg(next + q))
            if (q > last && q < best) best = q;
          if (best == 0x7fffffff) break;
          f4_add(d, ldg_cached(G4 + (int64_t)best * rm.cv + rm.c4));
          last = best;
        }
      }
    }
    return d;
  };
  auto emit = [&](int64_t e, const float4& a, const float4& b, const float4& d) {
    float gy[4], n[4], o[4];
    gn_gy(a, d, cf.sc, cf.of, cf.nm, cf.ni, thresh, inv_keep, seed_f, (uint64_t)e, relu, gy, n);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = cf.sc[i] * (gy[i] - n[i] * bmf[i]) - cof[i];
    stg_stream(of4 + e, make_float4(o[0], o[1], o[2], o[3]));
    gn_gy(b, d, cr.sc, cr.of, cr.nm, cr.ni, thresh, inv_keep, seed_r, (uint64_t)e, relu, gy, n);
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = cr.sc[i] * (gy[i] - n[i] * bmr[i]) - cor[i];
    stg_stream(or4 + e, make_float4(o[0], o[1], o[2], o[3]));
  };
  // two rows per thread and iteration: four streaming loads (+ two chain heads) in flight before any is consumed
  const int64_t stride = (int64_t)gridDim.x * rm.slots;
  for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += 2 * stride) {
    const int64_t r1 = r + stride;
    const bool two = r1 < M;
    const int64_t e0 = r * rm.cv + rm.c4, e1 = r1 * rm.cv + rm.c4;
    const float4 a0 = ldg_stream(xf4 + e0), b0 = ldg_stream(xr4 + e0);
    const float4 a1 = two ? ldg_stream(xf4 + e1) : f4_zero(), b1 = two ? ldg_stream(xr4 + e1) : f4_zero();
    const float4 d0 = chain_grad(r);
    const float4 d1 = two ? chain_grad(r1) : f4_zero();
    emit(e0, a0, b0, d0);
    if (two) emit(e1, a1, b1, d1);
  }
}

// out[c] = sum over CTAs of part[.][voff][c] for c < ncols (a warp per column)
__global__ void k_part_colsum_final(const double* __restrict__ part, int nparts, int nv, int voff, int C, int ncols,
                                    float* __restrict__ out) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= ncols) return;
  const double s = warp_part_sum(part, nparts, nv, voff, C, c);
  if ((threadIdx.x & 31) == 0) out[c] = (float)s;
}
// consts[4][C] = (P, Q, sc, of) of one GraphNorm branch for a consumer that applies its backward on the fly (twowl_pair_dw_gn):
//   dx = P*x + Q + sc*g_y,   P = -sc*ni*bm, Q = -(P*nm) - co   (the dense pass above, regrouped; g_y = 0 outside the selected rows)
//   and y = sc*x + of is the forward value the ReLU mask needs on the selected rows
__global__ void k_gn_bwd_consts(const float* __restrict__ stats, const float* __restrict__ weight, const float* __restrict__ bias,
                                const float* __restrict__ mean_scale, const float* __restrict__ sums, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float ni = stats[C + c], nm = mean_scale[c] * stats[c], sc = weight[c] * ni;
  const float P = -(sc * ni * sums[C + c]);
  out[c] = P;
  out[C + c] = -(P * nm) - sums[2 * C + c];
  out[2 * C + c] = sc;
  out[3 * C + c] = bias[c] - sc * nm;
}

// ---------------------------------------------------------------- column sum ---------------------
__global__ void __launch_bounds__(kNormThreads) k_colsum_partial(const float* __restrict__ x, int64_t M, int C,
                                                                 double* __restrict__ part) {
  const RowMap rm(C);
  float4 v[1] = {f4_zero()};
  ColFold<1> fold;
  if (rm.slot >= 0) {
    const float4* __restrict__ x4 = reinterpret_cast<const float4*>(x);
    for (int64_t r = (int64_t)blockIdx.x * rm.slots + rm.slot; r < M; r += (int64_t)gridDim.x * rm.slots) {
      f4_add(v[0], ldg_stream(x4 + r * rm.cv + rm.c4));
      fold.tick(v);
    }
    fold.flush(v);
  }
  cta_col_reduce_d<1>(rm, fold, part, C);
}
__global__ void k_colsum_final(const double* __restrict__ part, int nparts, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s = 0;
  for (int b = 0; b < nparts; ++b) s += part[(size_t)b * C + c];
  out[c] = (float)s;
}

static int norm_grid(int64_t M, int C) {
  const int slots = kNormThreads / (C >> 2);
  // at least 4 row iterations per CTA before adding CTAs; never more than 4 CTAs per SM
  int64_t g = cdiv(M, (int64_t)slots * 4);
  if (g > kNormMaxCtas) g = kNormMaxCtas;
  if (g < 1) g = 1;
  return (int)g;
}
// ColFold<nv>: nv x 4 doubles per thread
static size_t red_smem(int C, int nv) {
  (void)C;
  return (size_t)nv * 4 * kNormThreads * sizeof(double);
}
static int check_mc(const char* op, int64_t M, int C) {
  TW_CHECK_ARG(M >= 0 && C >= 4 && (C & 3) == 0 && C <= 1024, "%s: C=%d must be a multiple of 4 in [4,1024]", op, C);
  return 0;
}

}  // namespace twowl

using namespace twowl;

extern "C" size_t twowl_graphnorm_stats_workspace_bytes(int64_t M, int32_t C) {
  (void)M;
  return align_up((size_t)kNormMaxCtas * 2 * (size_t)C * sizeof(double));
}

extern "C" int twowl_graphnorm_stats(const float* x, int64_t M, int32_t C, const float* mean_scale, float eps, float* stats,
                                     void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_mc("graphnorm_stats", M, C)) return rc;
  TW_CHECK_ARG(M > 0, "graphnorm_stats: needs at least one row");
  TW_CHECK_ARG(aligned16(x), "graphnorm_stats: x must be 16-byte aligned");
  TW_CHECK_WS(ws_bytes, twowl_graphnorm_stats_workspace_bytes(M, C));
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = norm_grid(M, C);
  k_gn_stats_partial<<<grid, kNormThreads, red_smem(C, 2), s>>>(x, M, C, (double*)ws);
  k_gn_stats_final<<<(int)cdiv(C, 128), 128, 0, s>>>((const double*)ws, grid, x, M, C, mean_scale, eps, stats);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_graphnorm_apply(const float* x, int64_t M, int32_t C, const float* stats, const float* weight,
                                     const float* bias, const float* mean_scale, float p_drop, uint64_t seed, int32_t relu,
                                     const float* addend, float* out, void* stream) {
  if (int rc = check_mc("graphnorm_apply", M, C)) return rc;
  TW_CHECK_ARG(aligned16(x) && aligned16(out) && aligned16(addend), "graphnorm_apply: x/out/addend must be 16-byte aligned");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "graphnorm_apply: dropout p=%f outside [0,1)", p_drop);
  if (M == 0) return 0;
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  k_gn_apply<<<norm_grid(M, C), kNormThreads, 0, (cudaStream_t)stream>>>(x, M, C, stats, weight, bias, mean_scale, thresh,
                                                                        1.f / (1.f - p_drop), seed, relu, addend, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_graphnorm_bwd_workspace_bytes(int64_t M, int32_t C) {
  (void)M;
  return align_up((size_t)kNormMaxCtas * 2 * (size_t)C * sizeof(double)) + align_up(3 * (size_t)C * sizeof(float));
}

extern "C" int twowl_graphnorm_bwd(const float* x, const float* dout, int64_t M, int32_t C, const float* stats,
                                   const float* weight, const float* bias, const float* mean_scale, float p_drop, uint64_t seed,
                                   int32_t relu, float* dx, float* dparams, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_mc("graphnorm_bwd", M, C)) return rc;
  TW_CHECK_ARG(M > 0, "graphnorm_bwd: needs at least one row");
  TW_CHECK_ARG(aligned16(x) && aligned16(dout) && aligned16(dx), "graphnorm_bwd: x/dout/dx must be 16-byte aligned");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "graphnorm_bwd: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_graphnorm_bwd_workspace_bytes(M, C));
  cudaStream_t s = (cudaStream_t)stream;
  Carver c(ws);
  double* part = c.take<double>((size_t)kNormMaxCtas * 2 * C);
  float* sums = c.take<float>(3 * (size_t)C);
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  const float inv_keep = 1.f / (1.f - p_drop);
  const int grid = norm_grid(M, C);
  k_gn_bwd_partial<<<grid, kNormThreads, red_smem(C, 2), s>>>(x, dout, M, C, stats, weight, bias, mean_scale, thresh, inv_keep,
                                                              seed, relu, part);
  k_gn_bwd_final<<<(int)cdiv(C, 4), 128, 0, s>>>(part, grid, 2, 0, M, C, stats, weight, mean_scale, sums, dparams);
  k_gn_bwd_dx<<<grid, kNormThreads, 0, s>>>(x, dout, M, C, stats, weight, bias, mean_scale, thresh, inv_keep, seed, relu, sums,
                                            dx);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_colsum_workspace_bytes(int64_t M, int32_t C) {
  (void)M;
  return align_up((size_t)kNormMaxCtas * (size_t)C * sizeof(double));
}

extern "C" int twowl_colsum(const float* x, int64_t M, int32_t C, float* out, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_mc("colsum", M, C)) return rc;
  TW_CHECK_ARG(aligned16(x), "colsum: x must be 16-byte aligned");
  TW_CHECK_WS(ws_bytes, twowl_colsum_workspace_bytes(M, C));
  cudaStream_t s = (cudaStream_t)stream;
  if (M == 0) {
    TW_CUDA(cudaMemsetAsync(out, 0, (size_t)C * sizeof(float), s));
    return 0;
  }
  const int grid = norm_grid(M, C);
  k_colsum_partial<<<grid, kNormThreads, red_smem(C, 1), s>>>(x, M, C, (double*)ws);
  k_colsum_final<<<(int)cdiv(C, 128), 128, 0, s>>>((const double*)ws, grid, C, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_graphnorm_apply2(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                                      const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                      const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                                      int32_t relu, float* out, void* stream) {
  if (int rc = check_mc("graphnorm_apply2", M, C)) return rc;
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(out), "graphnorm_apply2: 16-byte alignment required");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "graphnorm_apply2: dropout p=%f outside [0,1)", p_drop);
  if (M == 0) return 0;
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  k_gn_apply2<<<norm_grid(M, C), kNormThreads, 0, (cudaStream_t)stream>>>(xf, xr, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr,
                                                                         thresh, 1.f / (1.f - p_drop), seed_f, seed_r, relu, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_gn2_readout_fwd(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                                     const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                     const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                                     int32_t relu, const int64_t* idx, int64_t sidx, int64_t L, const float* w, const float* b,
                                     float* pred, void* stream) {
  if (int rc = check_mc("gn2_readout_fwd", M, C)) return rc;
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(w), "gn2_readout_fwd: 16-byte alignment required");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "gn2_readout_fwd: dropout p=%f outside [0,1)", p_drop);
  if (L <= 0) return 0;
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  TW_CUDA(cudaMemsetAsync(pred, 0, (size_t)L * sizeof(float), (cudaStream_t)stream));   // logits of a masked tail (kMaskedTail)
#define TW_RO_ARGS xf, xr, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh, 1.f / (1.f - p_drop), seed_f, seed_r, relu, idx, sidx, L, w, b, pred
  cudaStream_t s = (cudaStream_t)stream;
  const int cv = C >> 2;
  if (cv <= 8)
    k_gn2_readout_fwd_g<8><<<grid_for(L, (kNormThreads / 32) * 4 * 2, 8), kNormThreads, 0, s>>>(TW_RO_ARGS);
  else if (cv <= 16)
    k_gn2_readout_fwd_g<16><<<grid_for(L, (kNormThreads / 32) * 2 * 2, 8), kNormThreads, 0, s>>>(TW_RO_ARGS);
  else if (cv <= 32)
    k_gn2_readout_fwd_g<32><<<grid_for(L, (kNormThreads / 32) * 2, 8), kNormThreads, 0, s>>>(TW_RO_ARGS);
  else
    k_gn2_readout_fwd<<<grid_for(L, kNormThreads / 32, 8), kNormThreads, 0, s>>>(TW_RO_ARGS);
#undef TW_RO_ARGS
  TW_LAUNCH_CHECK();
  return 0;
}

// everything of the fused GraphNorm-pair + readout backward except the dense dx pass
// rows: everything that touches the selected positions (per-position gradients G, chains, per-CTA column partials);
// finish: the column sums -> parameter gradients and the `sums` vectors the dense pass needs. M_stat = number of rows the
// GraphNorm statistics were taken over (= M on one GPU, the global row count when the pair table is row-sharded).
static int gn2_prepare_rows(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f, const float* stats_r,
                            const float* wf, const float* bf, const float* mf, const float* wr, const float* br, const float* mr,
                            uint32_t thresh, float inv_keep, uint64_t seed_f, uint64_t seed_r, int32_t relu, const int64_t* idx,
                            int64_t sidx, int64_t L, const float* w, const float* dpred, float* G, int32_t* head, int32_t* next,
                            double* part, int* nparts, cudaStream_t s) {
  const size_t l = (size_t)(L > 0 ? L : 1);
  TW_CUDA(cudaMemsetAsync(head, 0xFF, (size_t)M * sizeof(int32_t), s));
  const int grid_l = norm_grid(2 * (int64_t)l, C);
  k_gn2_readout_bwd_rows<<<grid_l, kNormThreads, red_smem(C, 6), s>>>(xf, xr, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh, inv_keep,
                                                                      seed_f, seed_r, relu, idx, sidx, L, w, dpred, G, part);
  if (L > 0) k_row_chains<<<grid_for(2 * L, kNormThreads), kNormThreads, 0, s>>>(idx, sidx, 2 * L, M, head, next);
  TW_LAUNCH_CHECK();
  *nparts = grid_l;
  return 0;
}
static int gn2_prepare_finish(const double* part, int nparts, int64_t M_stat, int32_t C, const float* stats_f, const float* stats_r,
                              const float* wf, const float* mf, const float* wr, const float* mr, float* sums_f, float* sums_r,
                              float* dparams_f, float* dparams_r, float* dw, float* db, cudaStream_t s) {
  k_gn_bwd_final<<<(int)cdiv(C, 4), 128, 0, s>>>(part, nparts, 6, 0, M_stat, C, stats_f, wf, mf, sums_f, dparams_f);
  k_gn_bwd_final<<<(int)cdiv(C, 4), 128, 0, s>>>(part, nparts, 6, 2, M_stat, C, stats_r, wr, mr, sums_r, dparams_r);
  k_part_colsum_final<<<(int)cdiv(C, 4), 128, 0, s>>>(part, nparts, 6, 4, C, C, dw);
  k_part_colsum_final<<<1, 32, 0, s>>>(part, nparts, 6, 5, C, 1, db);
  TW_LAUNCH_CHECK();
  return 0;
}
extern "C" size_t twowl_gn2_readout_bwd_workspace_bytes(int64_t M, int64_t L, int32_t C) {
  const size_t l = (size_t)(L > 0 ? L : 1);
  return align_up(2 * l * (size_t)C * sizeof(float)) + align_up((size_t)(M > 0 ? M : 1) * sizeof(int32_t)) + align_up(2 * l * sizeof(int32_t)) +
         align_up((size_t)kNormMaxCtas * 6 * (size_t)C * sizeof(double)) + 2 * align_up(3 * (size_t)C * sizeof(float));
}

extern "C" int twowl_gn2_readout_bwd(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                                     const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                     const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                                     int32_t relu, const int64_t* idx, int64_t sidx, int64_t L, const float* w, const float* dpred,
                                     float* dxf, float* dxr, float* dparams_f, float* dparams_r, float* dw, float* db, void* ws,
                                     size_t ws_bytes, void* stream) {
  if (int rc = check_mc("gn2_readout_bwd", M, C)) return rc;
  TW_CHECK_ARG(M > 0 && M < 0x7fffffffLL && L >= 0 && 2 * L < 0x7fffffffLL, "gn2_readout_bwd: sizes out of range");
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(dxf) && aligned16(dxr) && aligned16(w),
               "gn2_readout_bwd: 16-byte alignment required");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "gn2_readout_bwd: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_gn2_readout_bwd_workspace_bytes(M, L, C));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t l = (size_t)(L > 0 ? L : 1);
  Carver c(ws);
  float* G = c.take<float>(2 * l * C);
  int32_t* head = c.take<int32_t>((size_t)M);
  int32_t* next = c.take<int32_t>(2 * l);
  double* part = c.take<double>((size_t)kNormMaxCtas * 6 * C);
  float* sums_f = c.take<float>(3 * (size_t)C);
  float* sums_r = c.take<float>(3 * (size_t)C);
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  const float inv_keep = 1.f / (1.f - p_drop);
  int nparts = 0;
  if (int rc = gn2_prepare_rows(xf, xr, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh, inv_keep, seed_f, seed_r, relu, idx, sidx,
                                L, w, dpred, G, head, next, part, &nparts, s))
    return rc;
  if (int rc = gn2_prepare_finish(part, nparts, M, C, stats_f, stats_r, wf, mf, wr, mr, sums_f, sums_r, dparams_f, dparams_r, dw, db, s))
    return rc;
  k_gn_bwd2_dx_rows<<<norm_grid(M, C), kNormThreads, 0, s>>>(xf, xr, G, head, next, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh,
                                                             inv_keep, seed_f, seed_r, relu, sums_f, sums_r, dxf, dxr);
  TW_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------- backward halves ------------------
// The pair-layer backwards split at their column reductions: the first half stops at raw double sums over the caller's rows,
// a row-sharded caller adds them over the ranks (one all-reduce of a few KB), and the second half runs on the global sums. One
// GPU calls the halves back to back: the second half's warp_part_sum over nparts = 1 returns each sum unchanged, so the result
// is bit for bit that of one fused reduction.

// colsums[v][c] = sum over CTAs of part[.][v][c] (a warp per (v, c), fixed order)
__global__ void k_part_reduce_raw(const double* __restrict__ part, int nparts, int nv, int C, double* __restrict__ out) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= nv * C) return;
  const double s = warp_part_sum(part, nparts, nv, i / C, C, i % C);
  if ((threadIdx.x & 31) == 0) out[i] = s;
}

__global__ void k_gn_stats_from_moments(const double* __restrict__ mom, int64_t M, int C, const float* __restrict__ mean_scale,
                                        float eps, float* __restrict__ stats) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = mom[c] / (double)M;
  double var = mom[C + c] / (double)M - mean * mean;
  if (var < 0) var = 0;
  const double a = (double)mean_scale[c];
  stats[c] = (float)mean;
  stats[C + c] = (float)(1.0 / sqrt(var + (1.0 - a) * (1.0 - a) * mean * mean + (double)eps));
}

extern "C" int twowl_graphnorm_stats_from_moments(const double* moments, int64_t M, int32_t C, const float* mean_scale, float eps,
                                                  float* stats, void* stream) {
  if (int rc = check_mc("graphnorm_stats_from_moments", M, C)) return rc;
  TW_CHECK_ARG(M > 0 && moments && mean_scale && stats, "graphnorm_stats_from_moments: M > 0 and non-null pointers required");
  k_gn_stats_from_moments<<<(int)cdiv(C, 128), 128, 0, (cudaStream_t)stream>>>(moments, M, C, mean_scale, eps, stats);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_gn2_readout_bwd_rows_workspace_bytes(int64_t M, int64_t L, int32_t C) {
  (void)M, (void)L;
  return align_up((size_t)kNormMaxCtas * 6 * (size_t)C * sizeof(double));
}

extern "C" int twowl_gn2_readout_bwd_rows(const float* xf, const float* xr, int64_t M, int32_t C, const float* stats_f,
                                          const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                          const float* br, const float* mr, float p_drop, uint64_t seed_f, uint64_t seed_r,
                                          int32_t relu, const int64_t* idx, int64_t sidx, int64_t L, const float* w,
                                          const float* dpred, float* G, int32_t* head, int32_t* next, double* colsums, void* ws,
                                          size_t ws_bytes, void* stream) {
  if (int rc = check_mc("gn2_readout_bwd_rows", M, C)) return rc;
  TW_CHECK_ARG(M > 0 && M < 0x7fffffffLL && L >= 0 && 2 * L < 0x7fffffffLL, "gn2_readout_bwd_rows: sizes out of range");
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(G) && aligned16(w) && head && next && colsums,
               "gn2_readout_bwd_rows: bad pointers");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "gn2_readout_bwd_rows: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_gn2_readout_bwd_rows_workspace_bytes(M, L, C));
  cudaStream_t s = (cudaStream_t)stream;
  double* part = (double*)ws;
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  int nparts = 0;
  if (int rc = gn2_prepare_rows(xf, xr, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh, 1.f / (1.f - p_drop), seed_f, seed_r, relu,
                                idx, sidx, L, w, dpred, G, head, next, part, &nparts, s))
    return rc;
  k_part_reduce_raw<<<(int)cdiv(6 * C, 4), 128, 0, s>>>(part, nparts, 6, C, colsums);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_gn2_readout_bwd_finish_workspace_bytes(int32_t C) { return 2 * align_up(3 * (size_t)C * sizeof(float)); }

extern "C" int twowl_gn2_readout_bwd_finish(const double* colsums, int64_t M_total, int32_t C, const float* stats_f,
                                            const float* stats_r, const float* wf, const float* bf, const float* mf, const float* wr,
                                            const float* br, const float* mr, float* consts, float* dparams_f, float* dparams_r,
                                            float* dw, float* db, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_mc("gn2_readout_bwd_finish", M_total, C)) return rc;
  TW_CHECK_ARG(M_total > 0 && colsums && consts && dparams_f && dparams_r && dw && db, "gn2_readout_bwd_finish: bad arguments");
  TW_CHECK_WS(ws_bytes, twowl_gn2_readout_bwd_finish_workspace_bytes(C));
  cudaStream_t s = (cudaStream_t)stream;
  Carver c(ws);
  float* sums_f = c.take<float>(3 * (size_t)C);
  float* sums_r = c.take<float>(3 * (size_t)C);
  if (int rc = gn2_prepare_finish(colsums, 1, M_total, C, stats_f, stats_r, wf, mf, wr, mr, sums_f, sums_r, dparams_f, dparams_r, dw, db, s))
    return rc;
  k_gn_bwd_consts<<<(int)cdiv(C, 128), 128, 0, s>>>(stats_f, wf, bf, mf, sums_f, C, consts);
  k_gn_bwd_consts<<<(int)cdiv(C, 128), 128, 0, s>>>(stats_r, wr, br, mr, sums_r, C, consts + 4 * (size_t)C);
  TW_LAUNCH_CHECK();
  return 0;
}

// GraphNorm backward of both branches of a non-last pair layer: _sums gives the raw fp64 column sums [4][C] = per branch
// (sum g_y, sum g_y*n) over the caller's rows; _apply runs the finals on the (rank-summed) sums with the total row count M_total,
// then the dense dx pass over the caller's rows.
extern "C" size_t twowl_graphnorm_bwd2_sums_workspace_bytes(int64_t M, int32_t C) {
  (void)M;
  return align_up((size_t)kNormMaxCtas * 4 * (size_t)C * sizeof(double));
}

extern "C" int twowl_graphnorm_bwd2_sums(const float* xf, const float* xr, const float* dout, int64_t M, int32_t C,
                                         const float* stats_f, const float* stats_r, const float* wf, const float* bf,
                                         const float* mf, const float* wr, const float* br, const float* mr, float p_drop,
                                         uint64_t seed_f, uint64_t seed_r, int32_t relu, double* colsums, void* ws, size_t ws_bytes,
                                         void* stream) {
  if (int rc = check_mc("graphnorm_bwd2_sums", M, C)) return rc;
  TW_CHECK_ARG(M > 0 && colsums, "graphnorm_bwd2_sums: needs at least one row and an output");
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(dout), "graphnorm_bwd2_sums: 16-byte alignment required");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "graphnorm_bwd2_sums: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_graphnorm_bwd2_sums_workspace_bytes(M, C));
  cudaStream_t s = (cudaStream_t)stream;
  double* part = (double*)ws;
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  const int grid = norm_grid(M, C);
  k_gn_bwd2_partial<<<grid, kNormThreads, red_smem(C, 4), s>>>(xf, xr, dout, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh,
                                                               1.f / (1.f - p_drop), seed_f, seed_r, relu, part);
  k_part_reduce_raw<<<(int)cdiv(4 * C, 4), 128, 0, s>>>(part, grid, 4, C, colsums);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_graphnorm_bwd2_apply_workspace_bytes(int32_t C) { return 2 * align_up(3 * (size_t)C * sizeof(float)); }

extern "C" int twowl_graphnorm_bwd2_apply(const float* xf, const float* xr, const float* dout, int64_t M, int32_t C,
                                          const float* stats_f, const float* stats_r, const float* wf, const float* bf,
                                          const float* mf, const float* wr, const float* br, const float* mr, float p_drop,
                                          uint64_t seed_f, uint64_t seed_r, int32_t relu, const double* colsums, int64_t M_total,
                                          float* dxf, float* dxr, float* dparams_f, float* dparams_r, void* ws, size_t ws_bytes,
                                          void* stream) {
  if (int rc = check_mc("graphnorm_bwd2_apply", M, C)) return rc;
  TW_CHECK_ARG(M > 0 && M_total >= M && colsums, "graphnorm_bwd2_apply: needs rows, M_total >= M and the column sums");
  TW_CHECK_ARG(aligned16(xf) && aligned16(xr) && aligned16(dout) && aligned16(dxf) && aligned16(dxr),
               "graphnorm_bwd2_apply: 16-byte alignment required");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "graphnorm_bwd2_apply: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_graphnorm_bwd2_apply_workspace_bytes(C));
  cudaStream_t s = (cudaStream_t)stream;
  Carver c(ws);
  float* sums_f = c.take<float>(3 * (size_t)C);
  float* sums_r = c.take<float>(3 * (size_t)C);
  const uint32_t thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u;
  k_gn_bwd_final<<<(int)cdiv(C, 4), 128, 0, s>>>(colsums, 1, 4, 0, M_total, C, stats_f, wf, mf, sums_f, dparams_f);
  k_gn_bwd_final<<<(int)cdiv(C, 4), 128, 0, s>>>(colsums, 1, 4, 2, M_total, C, stats_r, wr, mr, sums_r, dparams_r);
  k_gn_bwd2_dx<<<norm_grid(M, C), kNormThreads, 0, s>>>(xf, xr, dout, M, C, stats_f, stats_r, wf, bf, mf, wr, br, mr, thresh,
                                                        1.f / (1.f - p_drop), seed_f, seed_r, relu, sums_f, sums_r, dxf, dxr);
  TW_LAUNCH_CHECK();
  return 0;
}
