// agg.cu - the segmented gather-reduce every TwoWL aggregation runs through, plus the gcn_norm degree.
//
// Replaces, on the hot path, PyG's gather -> scale -> scatter_add_ inside GCNConv.propagate
// (reference call sites TwoWL/model/model.py:73 node level, :77 pair level, both directions) and the
// autograd transposes of the same ops. HBM/L2-bound fp32 work: no tensor cores here.
//
// Layout: CSR by OUTPUT row (ptr int64[M+1], col int32[nnz]); features fp32 row-major [rows, C], C % 4 == 0.
// A row is owned by a group of G lanes (G = pow2 >= C/4, <= 32); each lane keeps VEC float4 accumulators.
// The group loads G col entries at once (coalesced), then broadcasts them one by one with shuffles and
// issues the 128-bit row gathers 4 deep. Sums run in CSR order (= the reference's column order, because the
// CSR is built by a STABLE sort) in registers: deterministic, no atomics on data.
//
// Power-law load balance: rows longer than TWOWL_LONG_ROW entries (hubs: max degree 62 745 on R-MAT 1M/16M)
// are listed once per CSR by twowl_seg_plan; they are cut into chunks of TWOWL_ROW_CHUNK entries that
// separate groups reduce into a partial buffer, and a third pass adds each row's partials in chunk order.
// The order in which long rows were listed (an integer atomic counter) never influences a result.
#include "common.cuh"

namespace twowl {

constexpr int kAggThreads = 256;

struct SegParams {
  const int64_t* ptr;
  const int32_t* col;
  int64_t M;
  const float* X;
  int C;
  int flip;
  int row_flip;
  int64_t row_lo, row_hi;      // output rows [row_lo, row_hi) only (a node block of a row-sharded job); the rest is untouched
  const float* src_scale;
  const uint8_t* skip_mask;
  const uint8_t* row_skip_mask;
  int skip_self;
  int self_mode;
  const float* dst_scale;
  const float* bias;
  const float* X2;
  const int32_t* mul_idx;
  float* out;
  int accumulate;
  int pair_sum;
  int x_shift;                 // 1: X holds ONE row per pair: entry s gathers X[s >> 1] (times X2: the row is already
                               // X[2k] + X[2k+1]; dual: the row is H[2k] = H[2k+1], the two directions' shared pair features)
  const uint8_t* entry_mask;
  // dual mode (MODE & 4): one pass over the 2-row blocks (s, s^1) feeds TWO outputs: out += src_scale[s] * X[s],
  // out2 += src_scale2[s^1] * X[s^1] - both directions of the pair layer's in-list sum, H read as 512-byte blocks
  const float* src_scale2;
  float* out2;
  float* partial2;
  const float* Xm;             // dual mode: the mates' rows come from this matrix instead of X (NULL = X)
  // long-row plan (all NULL/0 when the CSR has no plan)
  const int32_t* plan_counts;  // [0] = number of long rows, [1] = number of chunks
  const int32_t* long_row;     // CSR row of each long row
  const int32_t* long_base;    // first chunk slot of each long row
  const int32_t* chunk_owner;  // long-row slot of each chunk
  float* partial;              // [chunks, C]
};

// L2 policies of the gathers. Measured with ncu at R-MAT 1M/16M: every big seg_reduce launch moves 5.5-6.5 TB/s of DRAM traffic -
// the kernels are at the DRAM roofline for the bytes they touch, so the only lever is touching fewer. In the pair-init backward
// the rows of the [R, C] gradient are a stream (read twice, megabytes apart) while the rows of the per-NODE table x (268 MB,
// re-read deg(n) times) have reuse: stream = evict-first, table = evict-last (that launch: 44.8 -> 42.2 GB, 7.0 -> 6.7 ms).
// The same hints on the two-output passes (no table there) made them 10 % slower and are not used.
struct SegPolicies {
  uint64_t stream, keep;
  __device__ SegPolicies() {
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(stream));
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep));
  }
};
__device__ __forceinline__ float4 seg_ldg(const float4* p, uint64_t policy) {
  float4 r;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(policy));
  return r;
}

template <int G>
struct GroupCtx {
  int gl, gbase, cv;
  unsigned gmask;
  __device__ GroupCtx(int C) {
    const int lane = threadIdx.x & 31;
    gl = threadIdx.x % G;
    gbase = lane - gl;
    gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << gbase);
    cv = C >> 2;
  }
};

// acc += sum over entries [kb, ke) of the CSR feeding output row m.
// Software-pipelined two blocks deep so that no load is consumed in the iteration that issues it: while block b is
// gathered and accumulated, the col entries of block b+2 and the (col-dependent) scale / second-factor indices of
// block b+1 are in flight.
// MODE: 0 = plain gather, 1 = times X2[mul_idx], 3 = (X[s] + X[s^1]) times X2[mul_idx], 4 = dual (X[s] -> acc, X[s^1] -> acc2),
// 12 = dual over ONE row per pair (x_shift: X[s >> 1] is both X[s] and X[s^1], loaded once, added to acc and to acc2)
// (compile-time, so that the plain path keeps its registers for gathers in flight)
template <int G, int VEC, int MODE>
__device__ __forceinline__ void seg_accumulate(const SegParams& p, const GroupCtx<G>& g, const SegPolicies& pol, int64_t m, int64_t kb,
                                               int64_t ke, float4 (&acc)[VEC], float4 (&acc2)[(MODE & 4) ? VEC : 1]) {
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(p.X);
  const float4* __restrict__ X24 = reinterpret_cast<const float4*>(p.X2);
  const float4* __restrict__ Xm4 = ((MODE & 4) && p.Xm) ? reinterpret_cast<const float4*>(p.Xm) : X4;
  if (kb >= ke) return;
  auto load_col = [&](int64_t k0) -> int {
    const int64_t k = k0 + g.gl;
    return (k < ke && !(p.entry_mask && p.entry_mask[k])) ? __ldg(p.col + k) : -1;
  };
  // (col entry) -> source row (or -1 = dropped), its scale, optional second-factor row
  // m2_ carries the second-factor row (MODE & 1) or, bit-cast, the second scale (MODE & 4)
  auto stage = [&](int c, int& s_, float& w_, int& m2_) {
    s_ = -1, w_ = 0.f, m2_ = 0;
    if (c >= 0) {
      const int s = c ^ p.flip;
      const bool keep = !(p.skip_self && (int64_t)s == m) && !(p.skip_mask && p.skip_mask[c]);
      if (keep) {
        s_ = s;
        w_ = p.src_scale ? __ldg(p.src_scale + s) : 1.f;
        if (MODE & 1) m2_ = __ldg(p.mul_idx + c);
        if (MODE & 4) m2_ = __float_as_int(p.src_scale2 ? __ldg(p.src_scale2 + (s ^ 1)) : 1.f);
      }
    }
  };
  int c_b1 = load_col(kb + G);           // col of block b+1
  int s_mine, m2_mine;
  float w_mine;
  stage(load_col(kb), s_mine, w_mine, m2_mine);
  for (int64_t k0 = kb; k0 < ke; k0 += G) {
    const int c_b2 = load_col(k0 + 2 * G);
    int s_next, m2_next;
    float w_next;
    stage(c_b1, s_next, w_next, m2_next);
    const int cnt = (ke - k0 < G) ? (int)(ke - k0) : G;
    // UNR gathered rows are requested back to back (predicated 128-bit loads, no branches in between) before
    // any of them is consumed: the kernel lives on memory-level parallelism, not on occupancy
    constexpr int kLoads = 4;                     // rows in flight per lane and factor: occupancy beats deeper unrolling here
    constexpr int UNR = (VEC >= kLoads) ? 1 : (kLoads / VEC > G ? G : kLoads / VEC);
    for (int j0 = 0; j0 < cnt; j0 += UNR) {
      int sj[UNR], m2j[UNR];
      float wj[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int src_lane = g.gbase + ((j0 + u) & (G - 1));
        sj[u] = __shfl_sync(g.gmask, s_mine, src_lane);
        wj[u] = __shfl_sync(g.gmask, w_mine, src_lane);
        m2j[u] = __shfl_sync(g.gmask, m2_mine, src_lane);
        if (j0 + u >= cnt) sj[u] = -1;
      }
      float4 x[UNR][VEC], xm[(MODE & 6) ? UNR : 1][VEC], y[(MODE & 1) ? UNR : 1][VEC];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const int c4 = g.gl + v * G;
          const bool on = sj[u] >= 0 && c4 < g.cv;
          // with a second factor (pair-init backward): the [R, C] rows are a stream, the per-node table is what L2 should keep
          if (MODE & 1) {
            x[u][v] = on ? seg_ldg(X4 + (int64_t)((MODE & 2) ? sj[u] : (sj[u] >> p.x_shift)) * g.cv + c4, pol.stream) : f4_zero();
            if (MODE & 2) xm[u][v] = on ? seg_ldg(Xm4 + (int64_t)(sj[u] ^ 1) * g.cv + c4, pol.stream) : f4_zero();
            y[u][v] = on ? seg_ldg(X24 + (int64_t)m2j[u] * g.cv + c4, pol.keep) : f4_zero();
          } else if (MODE & 8) {
            x[u][v] = on ? ldg_cached(X4 + (int64_t)(sj[u] >> 1) * g.cv + c4) : f4_zero();
            xm[u][v] = x[u][v];
          } else {
            x[u][v] = on ? ldg_cached(X4 + (int64_t)sj[u] * g.cv + c4) : f4_zero();
            if (MODE & 6) xm[u][v] = on ? ldg_cached(Xm4 + (int64_t)(sj[u] ^ 1) * g.cv + c4) : f4_zero();
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        if (sj[u] >= 0) {
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            float4 t = x[u][v];
            if (MODE & 2) f4_add(t, xm[u][v]);
            if (MODE & 1) t = f4_mul(t, y[u][v]);
            f4_fma(acc[v], wj[u], t);
            if (MODE & 4) f4_fma(acc2[v], __int_as_float(m2j[u]), xm[u][v]);
          }
        }
      }
    }
    s_mine = s_next, w_mine = w_next, m2_mine = m2_next;
    c_b1 = c_b2;
  }
}

// out[m] = dst_scale*acc (+ self-loop term) (+ bias) (+ previous out)
template <int G, int VEC>
__device__ __forceinline__ void seg_finalize(const SegParams& p, const GroupCtx<G>& g, int64_t m, const float4 (&acc)[VEC]) {
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(p.X);
  const float ds = p.dst_scale ? p.dst_scale[m] : 1.f;
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    const int c4 = g.gl + v * G;
    if (c4 < g.cv) {
      float4 o = make_float4(ds * acc[v].x, ds * acc[v].y, ds * acc[v].z, ds * acc[v].w);
      if (p.self_mode == 1) f4_fma(o, ds * ds, ldg_cached(X4 + m * g.cv + c4));
      if (p.bias) f4_add(o, __ldg(reinterpret_cast<const float4*>(p.bias) + c4));
      float4* dst = reinterpret_cast<float4*>(p.out) + m * g.cv + c4;
      if (p.accumulate) f4_add(o, *dst);
      *dst = o;
    }
  }
}

// dual mode: the second output takes no epilogue terms
template <int G, int VEC>
__device__ __forceinline__ void seg_store2(const SegParams& p, const GroupCtx<G>& g, int64_t m, const float4 (&acc2)[VEC]) {
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    const int c4 = g.gl + v * G;
    if (c4 < g.cv) reinterpret_cast<float4*>(p.out2)[m * g.cv + c4] = acc2[v];
  }
}

// pass 1: one group per row, rows dealt round-robin to groups; long rows (if planned) are left to pass 2/3
template <int G, int VEC, int MODE>
__global__ void __launch_bounds__(kAggThreads) k_seg_rows(const SegParams p) {
  constexpr int kGroupsPerCta = kAggThreads / G;
  const GroupCtx<G> g(p.C);
  const SegPolicies pol;
  const int64_t group0 = (int64_t)blockIdx.x * kGroupsPerCta + threadIdx.x / G;
  const int64_t ngroups = (int64_t)gridDim.x * kGroupsPerCta;
  auto row_range = [&](int64_t m_, int64_t& kb_, int64_t& ke_, bool& masked_) {
    kb_ = 0, ke_ = 0, masked_ = false;
    const int64_t r = m_ ^ (int64_t)p.row_flip;
    if (m_ < p.M && r < p.M) {
      kb_ = __ldg(p.ptr + r);
      ke_ = __ldg(p.ptr + r + 1);
      masked_ = p.row_skip_mask && p.row_skip_mask[r];
    }
  };
  int64_t kb_n, ke_n;
  bool masked_n;
  row_range(p.row_lo + group0, kb_n, ke_n, masked_n);
  for (int64_t m = p.row_lo + group0; m < p.row_hi; m += ngroups) {
    const int64_t kb = kb_n;
    int64_t ke = ke_n;
    const bool masked = masked_n;
    row_range(m + ngroups, kb_n, ke_n, masked_n);  // next row's range is in flight while this row is reduced
    if (p.plan_counts && ke - kb > TWOWL_LONG_ROW) continue;  // handled by k_seg_chunks + k_seg_long
    if (masked) ke = kb;
    float4 acc[VEC], acc2[(MODE & 4) ? VEC : 1];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = f4_zero();
#pragma unroll
    for (int v = 0; v < ((MODE & 4) ? VEC : 1); ++v) acc2[v] = f4_zero();
    seg_accumulate<G, VEC, MODE>(p, g, pol, m, kb, ke, acc, acc2);
    seg_finalize<G, VEC>(p, g, m, acc);
    if constexpr ((MODE & 4) != 0) seg_store2<G, VEC>(p, g, m, acc2);
  }
}

// pass 2: one group per chunk of a long row -> raw partial sums
template <int G, int VEC, int MODE>
__global__ void __launch_bounds__(kAggThreads) k_seg_chunks(const SegParams p) {
  constexpr int kGroupsPerCta = kAggThreads / G;
  const GroupCtx<G> g(p.C);
  const SegPolicies pol;
  const int nchunks = p.plan_counts[1];
  const int64_t group0 = (int64_t)blockIdx.x * kGroupsPerCta + threadIdx.x / G;
  const int64_t ngroups = (int64_t)gridDim.x * kGroupsPerCta;
  for (int64_t ch = group0; ch < nchunks; ch += ngroups) {
    const int slot = p.chunk_owner[ch];
    const int64_t r = p.long_row[slot];
    const int64_t m = r ^ (int64_t)p.row_flip;
    if (m < p.row_lo || m >= p.row_hi) continue;
    const int64_t c = ch - p.long_base[slot];
    int64_t kb = p.ptr[r] + c * TWOWL_ROW_CHUNK;
    int64_t ke = kb + TWOWL_ROW_CHUNK < p.ptr[r + 1] ? kb + TWOWL_ROW_CHUNK : p.ptr[r + 1];
    if (p.row_skip_mask && p.row_skip_mask[r]) ke = kb;
    float4 acc[VEC], acc2[(MODE & 4) ? VEC : 1];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = f4_zero();
#pragma unroll
    for (int v = 0; v < ((MODE & 4) ? VEC : 1); ++v) acc2[v] = f4_zero();
    seg_accumulate<G, VEC, MODE>(p, g, pol, m, kb, ke, acc, acc2);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const int c4 = g.gl + v * G;
      if (c4 < g.cv) {
        reinterpret_cast<float4*>(p.partial)[ch * g.cv + c4] = acc[v];
        if constexpr ((MODE & 4) != 0) reinterpret_cast<float4*>(p.partial2)[ch * g.cv + c4] = acc2[v];
      }
    }
  }
}

// pass 3: partials of a long row added in a FIXED order, then the usual epilogue. Rows of up to kLongWide chunks: one lane
// group per row, chunk order. Longer rows (hubs: 980 chunks at degree 62 745; the embedding backward's "degree 1" row has
// thousands) would serialise thousands of dependent adds in one group, so a whole CTA takes the row: group j adds chunks
// j, j + n, j + 2n, ... in order, and the groups' sums are combined through shared memory in group order - a function of the
// chunk count only, hence still deterministic.
constexpr int kLongWide = 32;
template <int G, int VEC, bool DUAL>
__global__ void __launch_bounds__(kAggThreads) k_seg_long(const SegParams p) {
  constexpr int kGroupsPerCta = kAggThreads / G;
  const GroupCtx<G> g(p.C);
  const int nlong = p.plan_counts[0];
  const int gid = threadIdx.x / G;
  const int64_t group0 = (int64_t)blockIdx.x * kGroupsPerCta + gid;
  const int64_t ngroups = (int64_t)gridDim.x * kGroupsPerCta;
  auto chunks_of = [&](int64_t r) { return (p.ptr[r + 1] - p.ptr[r] + TWOWL_ROW_CHUNK - 1) / TWOWL_ROW_CHUNK; };
  // the chunk partials of a row are added in DOUBLE: a hub's row has ~1000 of them (degree 62 745), the "degree 1" row of the
  // embedding backward thousands, and an fp32 chain of that length would put ~sqrt(n) * 2^-24 of relative error into every
  // per-node sum that feeds all pairs centred on the hub; the 64 entries inside a chunk stay an fp32 chain
  auto add_chunks = [&](int64_t base, int64_t c0, int64_t cstep, int64_t nch, float4 (&acc)[VEC], float4 (&acc2)[DUAL ? VEC : 1]) {
    double d[VEC][4], d2[DUAL ? VEC : 1][4];
#pragma unroll
    for (int v = 0; v < VEC; ++v) d[v][0] = d[v][1] = d[v][2] = d[v][3] = 0.0;
#pragma unroll
    for (int v = 0; v < (DUAL ? VEC : 1); ++v) d2[v][0] = d2[v][1] = d2[v][2] = d2[v][3] = 0.0;
    for (int64_t c = c0; c < nch; c += cstep) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const int c4 = g.gl + v * G;
        if (c4 < g.cv) {
          const float4 t = reinterpret_cast<const float4*>(p.partial)[(base + c) * g.cv + c4];
          d[v][0] += (double)t.x, d[v][1] += (double)t.y, d[v][2] += (double)t.z, d[v][3] += (double)t.w;
          if constexpr (DUAL) {
            const float4 u = reinterpret_cast<const float4*>(p.partial2)[(base + c) * g.cv + c4];
            d2[v][0] += (double)u.x, d2[v][1] += (double)u.y, d2[v][2] += (double)u.z, d2[v][3] += (double)u.w;
          }
        }
      }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = make_float4((float)d[v][0], (float)d[v][1], (float)d[v][2], (float)d[v][3]);
    if constexpr (DUAL) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc2[v] = make_float4((float)d2[v][0], (float)d2[v][1], (float)d2[v][2], (float)d2[v][3]);
    }
  };
  // (a) short lists: one group per row
  for (int64_t slot = group0; slot < nlong; slot += ngroups) {
    const int64_t r = p.long_row[slot];
    const int64_t nch = chunks_of(r);
    if (nch > kLongWide || (r ^ (int64_t)p.row_flip) < p.row_lo || (r ^ (int64_t)p.row_flip) >= p.row_hi) continue;
    float4 acc[VEC], acc2[DUAL ? VEC : 1];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = f4_zero();
#pragma unroll
    for (int v = 0; v < (DUAL ? VEC : 1); ++v) acc2[v] = f4_zero();
    add_chunks(p.long_base[slot], 0, 1, nch, acc, acc2);
    const int64_t m = r ^ (int64_t)p.row_flip;
    seg_finalize<G, VEC>(p, g, m, acc);
    if constexpr (DUAL) seg_store2<G, VEC>(p, g, m, acc2);
  }
  // (b) long lists: one CTA per row
  extern __shared__ float4 seg_long_smem[];   // [kGroupsPerCta][DUAL ? 2 : 1][C / 4]
  for (int64_t slot = blockIdx.x; slot < nlong; slot += gridDim.x) {
    const int64_t r = p.long_row[slot];
    const int64_t nch = chunks_of(r);
    if (nch <= kLongWide || (r ^ (int64_t)p.row_flip) < p.row_lo || (r ^ (int64_t)p.row_flip) >= p.row_hi) continue;   // block-uniform
    float4 acc[VEC], acc2[DUAL ? VEC : 1];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = f4_zero();
#pragma unroll
    for (int v = 0; v < (DUAL ? VEC : 1); ++v) acc2[v] = f4_zero();
    add_chunks(p.long_base[slot], gid, kGroupsPerCta, nch, acc, acc2);
    constexpr int NV = DUAL ? 2 : 1;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const int c4 = g.gl + v * G;
      if (c4 < g.cv) {
        seg_long_smem[((size_t)gid * NV + 0) * g.cv + c4] = acc[v];
        if constexpr (DUAL) seg_long_smem[((size_t)gid * NV + 1) * g.cv + c4] = acc2[v];
      }
    }
    __syncthreads();
    if (gid == 0) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[v] = f4_zero();
#pragma unroll
      for (int v = 0; v < (DUAL ? VEC : 1); ++v) acc2[v] = f4_zero();
      for (int j = 0; j < kGroupsPerCta; ++j) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const int c4 = g.gl + v * G;
          if (c4 < g.cv) {
            f4_add(acc[v], seg_long_smem[((size_t)j * NV + 0) * g.cv + c4]);
            if constexpr (DUAL) f4_add(acc2[v], seg_long_smem[((size_t)j * NV + 1) * g.cv + c4]);
          }
        }
      }
      const int64_t m = r ^ (int64_t)p.row_flip;
      seg_finalize<G, VEC>(p, g, m, acc);
      if constexpr (DUAL) seg_store2<G, VEC>(p, g, m, acc2);
    }
    __syncthreads();
  }
}

template <int G, int VEC, int MODE>
static void launch_seg_mode(const SegParams& p, int64_t chunk_cap, int64_t long_cap, cudaStream_t s) {
  constexpr int kGroupsPerCta = kAggThreads / G;
  k_seg_rows<G, VEC, MODE><<<grid_for(p.row_hi - p.row_lo, kGroupsPerCta, 8), kAggThreads, 0, s>>>(p);
  if (p.plan_counts && chunk_cap > 0) {
    k_seg_chunks<G, VEC, MODE><<<grid_for(chunk_cap, kGroupsPerCta, 8), kAggThreads, 0, s>>>(p);
    const size_t lsm = (size_t)kGroupsPerCta * ((MODE & 4) ? 2 : 1) * (size_t)(p.C / 4) * sizeof(float4);
    if (lsm > 48 * 1024) cudaFuncSetAttribute(k_seg_long<G, VEC, (MODE & 4) != 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm);
    k_seg_long<G, VEC, (MODE & 4) != 0><<<grid_for(long_cap, kGroupsPerCta, 8), kAggThreads, lsm, s>>>(p);
  }
}
template <int G, int VEC>
static void launch_seg(const SegParams& p, int64_t chunk_cap, int64_t long_cap, cudaStream_t s) {
  if (p.out2 && p.x_shift) launch_seg_mode<G, VEC, 12>(p, chunk_cap, long_cap, s);
  else if (p.out2) launch_seg_mode<G, VEC, 4>(p, chunk_cap, long_cap, s);
  else if (!p.X2) launch_seg_mode<G, VEC, 0>(p, chunk_cap, long_cap, s);
  else if (!p.pair_sum) launch_seg_mode<G, VEC, 1>(p, chunk_cap, long_cap, s);
  else launch_seg_mode<G, VEC, 3>(p, chunk_cap, long_cap, s);
}

// ---------------------------------------------------------------- long-row plan ------------------
__global__ void __launch_bounds__(kAggThreads) k_plan_long(const int64_t* __restrict__ ptr, int64_t M, int32_t* __restrict__ counts,
                                                           int32_t* __restrict__ long_row, int32_t* __restrict__ long_base,
                                                           int32_t* __restrict__ chunk_owner) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t len = ptr[r + 1] - ptr[r];
    if (len > TWOWL_LONG_ROW) {
      const int nch = (int)((len + TWOWL_ROW_CHUNK - 1) / TWOWL_ROW_CHUNK);
      const int slot = atomicAdd(&counts[0], 1);   // listing order is free: results never depend on it
      const int base = atomicAdd(&counts[1], nch);
      long_row[slot] = (int32_t)r;
      long_base[slot] = base;
      for (int c = 0; c < nch; ++c) chunk_owner[base + c] = slot;
    }
  }
}

// deg[m] = 1 + #{k in row (m^row_flip) : (col[k]^flip) != m, !skip_mask[col[k]]}  ->  dinv = deg^-1/2
// one warp per row; integer counting, exact.
__global__ void __launch_bounds__(kAggThreads) k_gcn_dinv(const int64_t* __restrict__ ptr, const int32_t* __restrict__ col,
                                                          int64_t M, int flip, int row_flip,
                                                          const uint8_t* __restrict__ skip_mask,
                                                          const uint8_t* __restrict__ row_skip_mask, float* __restrict__ dinv) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * kAggThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kAggThreads) >> 5;
  for (int64_t m = warp0; m < M; m += nwarps) {
    const int64_t r = m ^ (int64_t)row_flip;
    int64_t kb = 0, ke = 0;
    if (r < M && !(row_skip_mask && row_skip_mask[r])) {
      kb = ptr[r];
      ke = ptr[r + 1];
    }
    // 8 x 32 entries per iteration, all loads issued before any is used: a hub row (62 745 entries) is one warp's serial
    // loop, and its latency chain was the whole kernel's tail (1.5 ms at R-MAT 1M/16M)
    int c = 0;
    constexpr int U = 8;
    for (int64_t k0 = kb; k0 < ke; k0 += 32 * U) {
      int cc[U];
      bool on[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t k = k0 + u * 32 + lane;
        on[u] = k < ke;
        cc[u] = on[u] ? __ldg(col + k) : 0;
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        c += (on[u] && ((int64_t)(cc[u] ^ flip) != m) && !(skip_mask && skip_mask[cc[u]])) ? 1 : 0;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if (lane == 0) dinv[m] = rsqrtf_exact((float)(c + 1));
  }
}

// the same count over the rows [row_lo, row_hi) of a cached CSR minus the entries a per-ENTRY mask removes:
// deg[m] = 1 + #{k in row m : !entry_mask[k], col[k] != m}
__global__ void __launch_bounds__(kAggThreads) k_gcn_dinv_entries(const int64_t* __restrict__ ptr, const int32_t* __restrict__ col,
                                                                  const uint8_t* __restrict__ entry_mask, int64_t row_lo,
                                                                  int64_t row_hi, float* __restrict__ dinv) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * kAggThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kAggThreads) >> 5;
  for (int64_t m = row_lo + warp0; m < row_hi; m += nwarps) {
    const int64_t kb = ptr[m], ke = ptr[m + 1];
    int c = 0;
    constexpr int U = 8;
    for (int64_t k0 = kb; k0 < ke; k0 += 32 * U) {
      int cc[U];
      bool on[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t k = k0 + u * 32 + lane;
        on[u] = k < ke && !(entry_mask && entry_mask[k]);
        cc[u] = on[u] ? __ldg(col + k) : 0;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) c += (on[u] && (int64_t)cc[u] != m) ? 1 : 0;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if (lane == 0) dinv[m] = rsqrtf_exact((float)(c + 1));
  }
}

}  // namespace twowl

using namespace twowl;

extern "C" int twowl_gcn_dinv(const int64_t* ptr, const int32_t* col, int64_t M, int32_t flip, int32_t row_flip,
                              const uint8_t* skip_mask, const uint8_t* row_skip_mask, float* dinv, void* stream) {
  TW_CHECK_ARG(M >= 0, "gcn_dinv: negative M");
  TW_CHECK_ARG(!(row_flip && (M & 1)), "gcn_dinv: row_flip needs an even row count");
  if (M == 0) return 0;
  k_gcn_dinv<<<grid_for(M, kAggThreads / 32, 8), kAggThreads, 0, (cudaStream_t)stream>>>(ptr, col, M, flip, row_flip, skip_mask,
                                                                                      row_skip_mask, dinv);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_gcn_dinv_entries(const int64_t* ptr, const int32_t* col, int64_t M, const uint8_t* entry_mask, int64_t row_lo,
                                      int64_t row_hi, float* dinv, void* stream) {
  TW_CHECK_ARG(M >= 0 && row_lo >= 0 && row_lo <= row_hi && row_hi <= M, "gcn_dinv_entries: rows [%lld, %lld) outside [0, %lld]",
               (long long)row_lo, (long long)row_hi, (long long)M);
  if (row_hi == row_lo) return 0;
  k_gcn_dinv_entries<<<grid_for(row_hi - row_lo, kAggThreads / 32, 8), kAggThreads, 0, (cudaStream_t)stream>>>(ptr, col, entry_mask,
                                                                                                          row_lo, row_hi, dinv);
  TW_LAUNCH_CHECK();
  return 0;
}

__global__ void __launch_bounds__(kAggThreads) k_gather_u8(const uint8_t* __restrict__ mask, const int32_t* __restrict__ ids, int64_t n,
                                                           uint8_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = mask[ids[i]];
}
extern "C" int twowl_gather_u8(const uint8_t* mask, const int32_t* ids, int64_t n, uint8_t* out, void* stream) {
  TW_CHECK_ARG(n >= 0, "gather_u8: negative n");
  if (n == 0) return 0;
  k_gather_u8<<<grid_for(n, kAggThreads, 8), kAggThreads, 0, (cudaStream_t)stream>>>(mask, ids, n, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t twowl_seg_plan_long_cap(int64_t nnz) { return nnz / TWOWL_LONG_ROW + 1; }
extern "C" int64_t twowl_seg_plan_chunk_cap(int64_t nnz) { return nnz / TWOWL_ROW_CHUNK + nnz / TWOWL_LONG_ROW + 2; }

extern "C" int twowl_seg_plan(const int64_t* ptr, int64_t M, int64_t nnz, int32_t* counts, int32_t* long_row, int32_t* long_base,
                              int32_t* chunk_owner, void* stream) {
  TW_CHECK_ARG(M >= 0 && nnz >= 0 && nnz < 0x7fffffffLL && M < 0x7fffffffLL, "seg_plan: sizes out of int32 range");
  cudaStream_t s = (cudaStream_t)stream;
  TW_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), s));
  if (M > 0) {
    k_plan_long<<<grid_for(M, kAggThreads), kAggThreads, 0, s>>>(ptr, M, counts, long_row, long_base, chunk_owner);
    TW_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" size_t twowl_sizeof_seg_args(void) { return sizeof(twowl_seg_args); }

extern "C" int twowl_seg_reduce(const twowl_seg_args* a, void* stream) {
  TW_CHECK_ARG(a != nullptr, "seg_reduce: null args");
  TW_CHECK_ARG(a->M >= 0 && a->C > 0 && (a->C & 3) == 0 && a->C <= 1024, "seg_reduce: C=%d must be a multiple of 4 in [4,1024]",
               a->C);
  TW_CHECK_ARG(aligned16(a->X) && aligned16(a->out) && aligned16(a->bias) && aligned16(a->X2) && aligned16(a->partial),
               "seg_reduce: feature pointers must be 16-byte aligned");
  TW_CHECK_ARG(!(a->row_flip && (a->M & 1)), "seg_reduce: row_flip needs an even row count");
  TW_CHECK_ARG((a->X2 == nullptr) == (a->mul_idx == nullptr), "seg_reduce: X2 and mul_idx go together");
  TW_CHECK_ARG(!a->pair_sum || a->X2 != nullptr || (a->pair_sum == 2 && a->out2),
               "seg_reduce: pair_sum is only built together with X2 (or, = 2, with the dual output)");
  TW_CHECK_ARG(!(a->pair_sum == 2 && a->X_mate), "seg_reduce: X_mate does not go with a one-row-per-pair X (pair_sum = 2)");
  TW_CHECK_ARG(a->pair_sum >= 0 && a->pair_sum <= 2, "seg_reduce: pair_sum = %d (0, 1 or 2)", a->pair_sum);
  TW_CHECK_ARG(!a->out2 || (!a->X2 && !a->flip && !a->row_flip && !a->accumulate && aligned16(a->out2) && aligned16(a->partial2)),
               "seg_reduce: dual output goes with a plain, unflipped, non-accumulating gather");
  const bool planned = a->plan_counts != nullptr;
  TW_CHECK_ARG(!planned || (a->long_row && a->long_base && a->chunk_owner && (a->partial || a->chunk_cap == 0) &&
                            (!a->out2 || a->partial2 || a->chunk_cap == 0)),
               "seg_reduce: incomplete long-row plan");
  TW_CHECK_ARG(a->row_begin >= 0 && a->row_end >= 0 && a->row_end <= a->M && (a->row_end == 0 || a->row_begin <= a->row_end),
               "seg_reduce: row range [%lld, %lld) outside [0, M]", (long long)a->row_begin, (long long)a->row_end);
  TW_CHECK_ARG(!(a->row_end && a->row_flip && ((a->row_begin | a->row_end) & 1)), "seg_reduce: a row range under row_flip needs even bounds");
  if (a->M == 0) return 0;
  SegParams p;
  p.row_lo = a->row_end ? a->row_begin : 0, p.row_hi = a->row_end ? a->row_end : a->M;   // row_end = 0: every row
  if (p.row_hi <= p.row_lo) return 0;
  p.ptr = a->ptr, p.col = a->col, p.M = a->M, p.X = a->X, p.C = a->C, p.flip = a->flip, p.row_flip = a->row_flip;
  p.src_scale = a->src_scale, p.skip_mask = a->skip_mask, p.row_skip_mask = a->row_skip_mask;
  p.skip_self = a->skip_self, p.self_mode = a->self_mode, p.dst_scale = a->dst_scale, p.bias = a->bias;
  p.X2 = a->X2, p.mul_idx = a->mul_idx, p.out = a->out, p.accumulate = a->accumulate, p.pair_sum = a->pair_sum == 1, p.x_shift = a->pair_sum == 2 ? 1 : 0, p.entry_mask = a->entry_mask;
  p.plan_counts = a->plan_counts, p.long_row = a->long_row, p.long_base = a->long_base, p.chunk_owner = a->chunk_owner;
  p.partial = a->partial;
  p.src_scale2 = a->src_scale2, p.out2 = a->out2, p.partial2 = a->partial2, p.Xm = a->X_mate;
  TW_CHECK_ARG(!a->X_mate || (a->out2 && aligned16(a->X_mate)), "seg_reduce: X_mate goes with the dual output");
  cudaStream_t s = (cudaStream_t)stream;
  const int cv = a->C >> 2;
  const int64_t cc = a->chunk_cap, lc = a->long_cap;
  if (cv <= 4) launch_seg<4, 1>(p, cc, lc, s);
  else if (cv <= 8) launch_seg<8, 1>(p, cc, lc, s);
  else if (cv <= 16) launch_seg<16, 1>(p, cc, lc, s);
  else if (cv <= 32) launch_seg<32, 1>(p, cc, lc, s);
  else if (cv <= 64) launch_seg<32, 2>(p, cc, lc, s);
  else if (cv <= 128) launch_seg<32, 4>(p, cc, lc, s);
  else launch_seg<32, 8>(p, cc, lc, s);
  TW_LAUNCH_CHECK();
  return 0;
}
