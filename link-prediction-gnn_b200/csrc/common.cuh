// common.cuh - shared host/device helpers for libtwowl_b200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/twowl.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libtwowl_b200 is written for sm_100a (B200) only"
#endif

namespace twowl {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

void set_error(const char* fmt, ...);

#define TW_CHECK_ARG(cond, ...)                 \
  do {                                          \
    if (!(cond)) {                              \
      ::twowl::set_error(__VA_ARGS__);          \
      return TWOWL_EINVAL;                      \
    }                                           \
  } while (0)

#define TW_CHECK_WS(have, need)                                                            \
  do {                                                                                     \
    if ((size_t)(have) < (size_t)(need)) {                                                 \
      ::twowl::set_error("workspace too small: have %zu need %zu", (size_t)(have), (size_t)(need)); \
      return TWOWL_ENOSPC;                                                                 \
    }                                                                                      \
  } while (0)

#define TW_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::twowl::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                                   \
    }                                                                                   \
  } while (0)

#define TW_LAUNCH_CHECK()                                                               \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      ::twowl::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                                   \
    }                                                                                   \
  } while (0)

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
// dropout threshold on the 32-bit hash for probability p
inline uint32_t drop_thresh(float p) {
  double t = (double)p * 4294967296.0;
  if (t < 0) t = 0;
  if (t > 4294967295.0) t = 4294967295.0;
  return (uint32_t)t;
}
inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// radix-sort key width: the fewest bits (1 to 32) that hold every value in [0, max_value]
inline int bits_for_value(int64_t max_value) {
  int b = 1;
  while (b < 32 && ((int64_t)1 << b) <= max_value) ++b;
  return b;
}

// grid for a grid-stride kernel: enough CTAs to cover `work_items` at `per_cta`, capped at a
// multiple of the SM count so every SM holds the same number of resident CTAs.
inline int grid_for(int64_t work_items, int64_t per_cta, int ctas_per_sm = 8) {
  int64_t g = cdiv(work_items, per_cta);
  int64_t cap = (int64_t)kNumSMs * ctas_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// Bump allocator over a caller-provided workspace.
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t n) {
    T* r = reinterpret_cast<T*>(base + off);
    off += align_up(n * sizeof(T));
    return r;
  }
};

#ifdef __CUDACC__
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  // read-once data: bypass L1 allocation (guide G13/G14)
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ldg_cached(const float4* p) { return __ldg(p); }
__device__ __forceinline__ void stg_stream(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
// deg^-1/2 with IEEE-rounded sqrt and divide (the reference's deg.pow(-0.5) on CPU), deg >= 1
__device__ __forceinline__ float rsqrtf_exact(float x) { return __fdiv_rn(1.f, __fsqrt_rn(x)); }
__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void f4_fma(float4& a, float s, const float4& x) {
  a.x = fmaf(s, x.x, a.x);
  a.y = fmaf(s, x.y, a.y);
  a.z = fmaf(s, x.z, a.z);
  a.w = fmaf(s, x.w, a.w);
}
__device__ __forceinline__ void f4_add(float4& a, const float4& x) {
  a.x += x.x;
  a.y += x.y;
  a.z += x.z;
  a.w += x.w;
}
__device__ __forceinline__ float4 f4_mul(const float4& a, const float4& b) {
  return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
}
// A seed argument with bit 63 set is not the seed but the ADDRESS (low 63 bits) of a device uint64 that holds it: a step
// captured as a CUDA graph bakes its scalar arguments in, so its dropout seeds live in device memory and are refreshed
// between replays (twowl_b200/graphed.py). Host-drawn seeds are below 2^62.
__device__ __forceinline__ uint64_t resolve_seed(uint64_t seed) {
  return (seed >> 63) ? __ldg(reinterpret_cast<const unsigned long long*>(seed & 0x7fffffffffffffffull)) : seed;
}
__device__ __forceinline__ uint32_t hash_u32(uint64_t seed, uint64_t idx) {
  // splitmix64 finaliser over (seed, element index): counter-based, so the backward regenerates the dropout mask.
  // `seed` is the VALUE: kernels resolve a tagged seed once at entry (resolve_seed), never per element.
  uint64_t z = idx + seed * 0x9E3779B97F4A7C15ull + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (uint32_t)(z >> 32);
}
// 1/(1-p) if element kept else 0
__device__ __forceinline__ float drop_scale(uint64_t seed, uint64_t idx, uint32_t thresh, float inv_keep) {
  return hash_u32(seed, idx) >= thresh ? inv_keep : 0.f;
}
__device__ __forceinline__ uint32_t auc_key(float x) {
  // ascending order-preserving map of IEEE-754 floats to uint32 (-0 and +0 share a key; NaNs sort last)
  if (x == 0.f) x = 0.f;
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float4 f4_shfl_xor(const float4& v, int m) {
  return make_float4(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m),
                     __shfl_xor_sync(0xffffffffu, v.z, m), __shfl_xor_sync(0xffffffffu, v.w, m));
}
#endif

// ---- primitives implemented in prims.cu (device-side building blocks, all on `stream`) ----------

// out[i] = sum_{j<i} in[j] for i in [0,n]; out has n+1 slots (out[n] = total). in == out allowed when
// both are int64. ws: scan_workspace_bytes(n).
size_t scan_workspace_bytes(int64_t n);
int scan_exclusive_i64(const int64_t* in, int64_t* out, int64_t n, void* ws, cudaStream_t s);

// Stable LSD radix sort of (key, val) uint32 pairs on the low `bits` bits of key. Result ends in
// (keys_out, vals_out); keys_in/vals_in are clobbered. ws: radix_workspace_bytes(n).
size_t radix_workspace_bytes(int64_t n);
int radix_sort_pairs(uint32_t* keys_in, uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, int64_t n,
                     int bits, void* ws, cudaStream_t s);

// ---- TMA tensor map of a row-major fp32 [rows, cols] matrix (prims.cu): boxes of box_cols x box_rows elements.
// cuTensorMapEncodeTiled is reached through the runtime's driver entry point, so libcuda is not linked.
// ld = row pitch in elements (0 = cols: a dense matrix); a column block of a wider matrix is base = X + c0, cols = width, ld = X's width.
int make_tmap_2d_f32(CUtensorMap* tm, const float* base, int64_t rows, int cols, int box_cols, int box_rows,
                     CUtensorMapSwizzle swizzle, int64_t ld = 0);

// ---- tensor-core linear layer: the pair_conv kernel with one source and no epilogue terms (pair_conv.cu) ----------------------------------------
// C[M,Nd] = A[M,Kd] * B^T with B[n][k] = W[n*Kd+k] (w_kn = 0) or W[k*Nd+n] (w_kn = 1); tcgen05 kind::tf32, 3xTF32.
bool linear_tc_supported(int Kd, int Nd);
int linear_tc(const float* A, const float* W, float* C, int64_t M, int Kd, int Nd, int w_kn, cudaStream_t s);

}  // namespace twowl
