// pair_conv.cu - the pair-level GCNConv of TwoWL/model/model.py:77 with its dense linear layer on tcgen05 tensor
// cores and the structured ("factorised") aggregation fused into the GEMM's epilogue:
//
//   out[r, :] = sum_{s < nsrc} rs_s[r] * (A_s[r, :] * B_s^T)  +  sum_{g < ngather} coef_g[r] * T_g[idx_g[r], :]  +  bias
//
//   forward, one direction d :  A = H, rs = selfw_d, B = W_d, gather (S_d, centre_d, dinv_d), bias_d, + column
//                               statistics of `out` for the GraphNorm that follows (no extra pass over out)
//   backward w.r.t. H        :  A = (dO_f, dO_r), rs = (selfw_f, selfw_r), B = (W_f^T, W_r^T), gathers
//                               ((dS_f W_f), node_f, dinv_f) and ((dS_r W_r), node_r, dinv_r)
//   plain linear             :  nsrc = 1, no scale, no gather
//
// One persistent CTA per SM, 12 warps, warp-specialised:
//   warp  0    TMA producer: one lane streams raw fp32 128-row tiles of A_s into a ring of shared-memory stages with
//                            cp.async.bulk.tensor (SWIZZLE_128B tensor map = the UMMA canonical K-major layout, L2
//                            evict-first), 2-3 tiles in flight per SM
//   warps 2-3  split       : lo = rn_tf32(x - trunc_tf32(x)) of a landed tile into a second buffer (smem -> smem). The tensor
//                            core TRUNCATES fp32 operands to tf32 (measured, tools/mma_probe.cu), so the raw tile IS
//                            the `hi` operand of the split-tf32 scheme and is never rewritten
//   warp  1    MMA issuer  : one lane issues 3 x Kd/8 tcgen05.mma kind::tf32 per source (lo*hi, hi*lo, hi*hi) into that
//                            source's TMEM accumulator (double buffered); tcgen05.commit releases the stages / publishes
//   warps 4-11 epilogue    : (4 TMEM lane quarters x 2 column halves) gathered rows requested before the accumulator
//                            is waited for; tcgen05.ld -> row scale, source sum -> per-warp smem transpose -> coalesced
//                            128-byte row segments: gather terms, bias, store, column sums (fp32 per tile -> double per
//                            CTA, fixed order)
// HBM-bound by design: 4*M*(nsrc*Kd + Nd) bytes + gathers for 6*M*Kd*Nd*nsrc tensor flop.
#include "common.cuh"

namespace twowl {

constexpr int kPcSplitWarps = 2;
constexpr int kPcEpilogueWarps = 8;
constexpr int kPcFirstSplit = 2;
constexpr int kPcFirstEpi = kPcFirstSplit + kPcSplitWarps;                    // 4
constexpr int kPcThreads = (kPcFirstEpi + kPcEpilogueWarps) * 32;            // 384: 12 warps -> up to 168 registers per thread
constexpr int kPcTileM = 128;
constexpr uint32_t kPcSlab = kPcTileM * 128u;  // 128 rows x 32 fp32 columns = one SWIZZLE_128B K-slab (16 KB)
constexpr int kPcGroup = 2;                    // pipeline unit: up to 2 K-slabs (one barrier round trip per 32 KB)
constexpr uint32_t kPcStage = kPcGroup * kPcSlab;
constexpr int kPcMaxStages = 4;                // raw-stage ring
constexpr int kPcMaxLo = 2;                    // lo-stage ring

struct ConvParams {
  const float* rs[2];
  const float* W[2];
  int w_kn[2];
  int nsrc;
  int64_t M;
  int Kd, Nd;          // full widths of A and out
  int Nsub, nsplit;    // output columns per CTA (multiple of 16) and the number of column windows
  const float* T[2];
  const int32_t* tidx[2];
  const float* tcoef[2];
  int ngather;
  const float* bias;
  float* out;
  int group;           // K-slabs per pipeline stage (1 or 2)
  double* stats_part;  // [gridDim.x][2][Nsub] column (sum, sum of squares) of this CTA's window of `out`, or NULL
  int tmem_cols;
  int stages;          // raw-stage ring depth (2..kPcMaxStages)
  int lo_stages;       // lo-stage ring depth (1..kPcMaxLo)
};

__device__ __forceinline__ uint32_t pc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t pc_desc(uint32_t saddr) {
  // K-major SWIZZLE_128B, 8-row groups 1024 B apart, descriptor version 1 (sm_100)
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)64 << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void pc_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void pc_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(pc_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void pc_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(pc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void pc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pc_tma_load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
          pc_smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(pc_smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void pc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(pc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void pc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void pc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void pc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void pc_proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void pc_tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// gathered table rows are the only data of this kernel with reuse: ask L2 to keep them (the streamed tiles are evict-first)
__device__ __forceinline__ float4 pc_ldg_keep(const float4* p, uint64_t policy) {
  float4 r;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(policy));
  return r;
}
__device__ __forceinline__ void pc_tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t pc_sw128(int r, int c) { return (uint32_t)(((r >> 3) << 10) + ((r & 7) << 7) + (((c ^ r) & 7) << 4)); }
// The tf32 split of the GEMM operands. The tensor core TRUNCATES fp32 operands to tf32 (tools/mma_probe.cu), so
//   A (streamed): the raw tile is read as hi = trunc_tf32(x) for free; the split warps add lo = rn_tf32(x - hi) in a second
//                 buffer (x - hi is exact, < 2^-10 |x|; rounding it to NEAREST instead of letting the tensor core truncate it
//                 halves the error and removes its bias: |x - hi - lo| <= 2^-21 |x|);
//   W (resident): hi = rn_tf32(w), lo = rn_tf32(w - hi): |w - hi - lo| <= 2^-22 |w|, |lo| <= 2^-11 |w|.
// Three products hi*hi + hi*lo + lo*hi are issued; the dropped lo*lo is <= 2^-21 |a*w|. Per product the relative error is
// <= 2^-21 + 2^-22 + 2^-21 = 1.25 * 2^-20, unbiased (round 1: 3 * 2^-20 with every term biased towards zero). A fourth
// product and a round-to-nearest hi written back in place were measured: 4x smaller GEMM error, no change of the end-to-end
// error (which is dominated by the conditioning of the fp32 chain, tools/diag_parity.py) and +11 % step time - not kept.
// round to nearest tf32 (ties away from zero, = cvt.rna.tf32.f32) with two integer-pipe instructions: half an ulp of the
// 10-bit mantissa added to the magnitude bits, the 13 low bits cleared (a carry into the exponent is the correct result). The
// cvt instruction itself issues on the quarter-rate conversion pipe, which the latency-bound split warps feel.
__device__ __forceinline__ float pc_rna(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
__device__ __forceinline__ float pc_lo(float x) { return pc_rna(x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u)); }
__device__ __forceinline__ void pc_split(const float4& v, float4& hi, float4& lo) {   // resident weights
  hi.x = pc_rna(v.x), hi.y = pc_rna(v.y), hi.z = pc_rna(v.z), hi.w = pc_rna(v.w);
  lo.x = pc_rna(v.x - hi.x), lo.y = pc_rna(v.y - hi.y), lo.z = pc_rna(v.z - hi.z), lo.w = pc_rna(v.w - hi.w);
}
// One lane of a converged warp. The single-thread instructions (TMA, tcgen05.mma / commit) are issued under this predicate
// with the WHOLE warp running the surrounding loop on warp-uniform values: the compiler then keeps descriptors and
// addresses in uniform registers and emits the UTCHMMA / UTMALDG back to back. Under a divergent `if (lane == 0)` every
// one of them is wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~16-30 instructions of serial latency per MMA),
// which made the issuing thread the bottleneck of the kernel.
__device__ __forceinline__ bool pc_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// ring position: slot and the parity of the round it is in
struct PcRing {
  int slot = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void next(int depth) {
    if (++slot == depth) slot = 0, phase ^= 1u;
  }
};

// CTA b works on column window b % nsplit of the tiles (b / nsplit) + j * (gridDim.x / nsplit): the CTAs that share a
// tile run side by side, so the re-reads of its A slabs are L2 hits.
// PSUM (compile time, its own instantiation - a runtime flag changed the register allocation of every other one and cost the
// forward launches 1 ms each): out has M/2 rows, out[k] = result[2k] + result[2k+1]
// APAIR (compile time, likewise; nsrc = 1): A has M/2 rows, one per pair, and output row r uses A row r >> 1 - the depth-1 pair
// layer's H, whose rows 2k / 2k+1 are the same bits (twowl_conv_args.a_pairs). The 64 pairs of a 128-row tile land as four
// 16-row boxes at rows 0 / 32 / 64 / 96 of the stage, so TMEM lanes 32q..32q+15 hold the products of pairs 16q..16q+15 and
// epilogue lane l of quarter q takes its row's values from lane l >> 1. Rows 16..31 of each quarter hold stale data whose
// products land in TMEM lanes nobody reads; the MMA, the epilogue's rows, gathers, stores and statistics are unchanged.
template <int NG, bool PSUM = false, bool APAIR = false>
__global__ void __launch_bounds__(kPcThreads, 1) k_pair_conv(const ConvParams p, const __grid_constant__ CUtensorMap tmA0,
                                                             const __grid_constant__ CUtensorMap tmA1) {
  extern __shared__ uint8_t pc_smem_raw[];
  // 1024-byte alignment by OFFSET from the shared array: a pointer rebuilt from an integer would be generic (LD.E / ST.E)
  uint8_t* smem = pc_smem_raw + ((1024u - (pc_smem_u32(pc_smem_raw) & 1023u)) & 1023u);
  const int Nd = p.Nd, Nsub = p.Nsub, Kd = p.Kd;
  const int KB = (Kd + 31) >> 5;                 // K-slabs per tile
  const int Nsp = (Nsub + 31) & ~31;             // TMEM columns per source accumulator (the epilogue reads 32-column blocks)
  const int S = p.stages, LS = p.lo_stages;
  const int G = KB > 1 ? p.group : 1;            // K-slabs per pipeline stage
  const uint32_t kStage = (uint32_t)G * kPcSlab;  // bytes per pipeline stage
  const uint32_t kBSlab = (uint32_t)Nsub * 128u;         // one K-slab of one of hi / lo of one source
  const uint32_t kBMat = (uint32_t)KB * kBSlab;
  uint8_t* Bs = smem;                                   // [nsrc][hi, lo][KB][Nsub rows x 128 B]
  uint8_t* As = Bs + (size_t)p.nsrc * 2 * kBMat;        // [S] raw stages of kPcGroup slabs
  uint8_t* Ls = As + (size_t)S * kStage;              // [LS] lo stages
  uint8_t* Es = Ls + (size_t)LS * kStage;             // [epilogue warp] 32 rows x 32 cols fp32 transpose buffer
  uint64_t* bars = reinterpret_cast<uint64_t*>(Es + kPcEpilogueWarps * 4096);
  uint64_t* raw_full = bars;                            // [S]  TMA -> split, MMA
  uint64_t* raw_empty = raw_full + kPcMaxStages;        // [S]  MMA -> TMA
  uint64_t* lo_full = raw_empty + kPcMaxStages;         // [LS] split -> MMA
  uint64_t* lo_empty = lo_full + kPcMaxLo;              // [LS] MMA -> split
  uint64_t* tfull = lo_empty + kPcMaxLo;                // [2]  MMA -> epilogue
  uint64_t* tempty = tfull + 2;                         // [2]  epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  double* red = reinterpret_cast<double*>(tempty + 4);  // [epilogue warps][2][Nsub] end-of-kernel reduction

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = (int)(blockIdx.x % p.nsplit), grp = (int)(blockIdx.x / p.nsplit), ngrp = (int)(gridDim.x / p.nsplit);
  const int n0 = split * Nsub;
  const int64_t ntiles = (p.M + kPcTileM - 1) / kPcTileM;
  const int64_t my_tiles = (ntiles > grp) ? (ntiles - grp + ngrp - 1) / ngrp : 0;

  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(pc_smem_u32(tmem_slot)), "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int s = 0; s < kPcMaxStages; ++s) {
      pc_mbar_init(&raw_full[s], 1);
      pc_mbar_init(&raw_empty[s], 1);
    }
    for (int s = 0; s < kPcMaxLo; ++s) {
      pc_mbar_init(&lo_full[s], kPcSplitWarps * 32);
      pc_mbar_init(&lo_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      pc_mbar_init(&tfull[a], 1);
      pc_mbar_init(&tempty[a], kPcEpilogueWarps * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA0)) : "memory");
    if (p.nsrc > 1) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA1)) : "memory");
  }
  // resident weights of this CTA's column window: hi/lo split in the canonical layout (K-slab = 32 k-values, Nsub rows of
  // 128 bytes); rows beyond Nd and k beyond Kd are zero
  for (int s = 0; s < p.nsrc; ++s) {
    const float* __restrict__ W = (s == 0) ? p.W[0] : p.W[1];
    const int w_kn = (s == 0) ? p.w_kn[0] : p.w_kn[1];
    uint8_t* Bhi = Bs + (size_t)s * 2 * kBMat;
    uint8_t* Blo = Bhi + kBMat;
    const int K4p = KB * 8;
    for (int i = tid; i < Nsub * K4p; i += kPcThreads) {
      const int n = i / K4p, k4 = i % K4p;
      const int gn = n0 + n, k = k4 * 4;
      float4 v = f4_zero();
      if (gn < Nd && k < Kd) {
        if (!w_kn) {
          v = __ldg(reinterpret_cast<const float4*>(W + (size_t)gn * Kd + k));
        } else {
          v.x = __ldg(W + (size_t)(k + 0) * Nd + gn);
          v.y = __ldg(W + (size_t)(k + 1) * Nd + gn);
          v.z = __ldg(W + (size_t)(k + 2) * Nd + gn);
          v.w = __ldg(W + (size_t)(k + 3) * Nd + gn);
        }
      }
      float4 hi, lo;
      pc_split(v, hi, lo);
      const uint32_t off = (uint32_t)(k4 >> 3) * kBSlab + pc_sw128(n, k4 & 7);
      *reinterpret_cast<float4*>(Bhi + off) = hi;
      *reinterpret_cast<float4*>(Blo + off) = lo;
    }
  }
  if (p.stats_part)
    for (int i = tid; i < kPcEpilogueWarps * 2 * Nsub; i += kPcThreads) red[i] = 0.0;
  pc_proxy_fence();
  pc_fence_before();
  __syncthreads();
  pc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform

  if (warp == 0) {
    // ===================================================== TMA producer: stages in (tile, source, k-group) order
    // a tile streamed once is evict-first; with column windows the nsplit CTAs of a tile fetch it one after the other, so the
    // first fetch must stay in L2 for the others (evict-first made every window re-read its tile from DRAM: 27.5 GB read for
    // 15.4 GB of input at C = 128)
    uint64_t policy;
    if (p.nsplit > 1)
      asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(policy));
    else
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    PcRing r;
    for (int64_t ti = 0; ti < my_tiles; ++ti) {
      const int row0 = (int)((grp + ti * ngrp) * kPcTileM);
      for (int s = 0; s < p.nsrc; ++s) {
        const CUtensorMap* tm = s ? &tmA1 : &tmA0;
        for (int kb = 0; kb < KB; kb += G) {
          const int ns = KB - kb < G ? KB - kb : G;
          pc_mbar_wait(&raw_empty[r.slot], r.phase ^ 1u);
          if (pc_elect_one()) {
            if constexpr (APAIR) {
              pc_mbar_expect_tx(&raw_full[r.slot], (uint32_t)ns * (kPcSlab / 2));
              for (int j = 0; j < ns; ++j)
                for (int q = 0; q < 4; ++q)
                  pc_tma_load_2d(As + (size_t)r.slot * kStage + (size_t)j * kPcSlab + q * 4096, tm, (kb + j) * 32, (row0 >> 1) + q * 16,
                                 &raw_full[r.slot], policy);
            } else {
              pc_mbar_expect_tx(&raw_full[r.slot], (uint32_t)ns * kPcSlab);
              for (int j = 0; j < ns; ++j)
                pc_tma_load_2d(As + (size_t)r.slot * kStage + (size_t)j * kPcSlab, tm, (kb + j) * 32, row0, &raw_full[r.slot], policy);
            }
          }
          __syncwarp();
          r.next(S);
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(Nsub >> 3) << 17) | ((uint32_t)(kPcTileM >> 4) << 24);
    PcRing r, l;
    for (int64_t ti = 0; ti < my_tiles; ++ti) {
      const int a = (int)(ti & 1);
      pc_mbar_wait(&tempty[a], (uint32_t)(((ti >> 1) & 1) ^ 1));
      pc_fence_after();
      for (int s = 0; s < p.nsrc; ++s) {
        const uint32_t tacc = tmem_base + (uint32_t)(a * (p.tmem_cols >> 1) + s * Nsp);
        const uint32_t Bhi = pc_smem_u32(Bs + (size_t)s * 2 * kBMat), Blo = Bhi + kBMat;
        uint32_t acc = 0;
        for (int kb = 0; kb < KB; kb += G) {
          const int ns = KB - kb < G ? KB - kb : G;
          pc_mbar_wait(&raw_full[r.slot], r.phase);
          pc_mbar_wait(&lo_full[l.slot], l.phase);
          pc_fence_after();
          // descriptors advance by byte offset >> 4 in their low word (no carry out of the 14-bit address field: smem < 256 KB)
          const uint64_t Ahi = pc_desc(pc_smem_u32(As) + (uint32_t)r.slot * kStage), Alo = pc_desc(pc_smem_u32(Ls) + (uint32_t)l.slot * kStage);
          const uint64_t bhi = pc_desc(Bhi + (uint32_t)kb * kBSlab), blo = pc_desc(Blo + (uint32_t)kb * kBSlab);
          const uint32_t bstep = kBSlab >> 4;
          if (pc_elect_one()) {
            if (ns == 1 && Kd - kb * 32 >= 32) {
              // one full slab per stage (the 16 KB ring of the wide two-source launches)
#pragma unroll
              for (int pass = 0; pass < 3; ++pass) {
                const uint64_t Ap = (pass == 0) ? Alo : Ahi;
                const uint64_t Bp = (pass == 1) ? blo : bhi;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  pc_mma(tacc, Ap + (uint64_t)(k * 2), Bp + (uint64_t)(k * 2), idesc, acc);
                  acc = 1;
                }
                if (pass == 0) pc_commit(&lo_empty[l.slot]);
              }
            } else if (ns == kPcGroup && Kd - kb * 32 >= kPcGroup * 32) {
              // full stage: 3 passes (lo*hi, hi*lo, hi*hi: small terms first - the accumulator's own truncation is relative to
              // its magnitude) x 2 slabs x 4 k-steps, back to back
#pragma unroll
              for (int pass = 0; pass < 3; ++pass) {
                const uint64_t Ap = (pass == 0) ? Alo : Ahi;
                const uint64_t Bp = (pass == 1) ? blo : bhi;
#pragma unroll
                for (int j = 0; j < kPcGroup; ++j) {
#pragma unroll
                  for (int k = 0; k < 4; ++k) {
                    pc_mma(tacc, Ap + (uint64_t)(j * (kPcSlab >> 4) + k * 2), Bp + (uint64_t)(j * bstep + k * 2), idesc, acc);
                    acc = 1;
                  }
                }
                if (pass == 0) pc_commit(&lo_empty[l.slot]);  // the lo stage is free once the first pass has read it
              }
            } else {
              for (int pass = 0; pass < 3; ++pass) {
                const uint64_t Ap = (pass == 0) ? Alo : Ahi;
                const uint64_t Bp = (pass == 1) ? blo : bhi;
                for (int j = 0; j < ns; ++j) {
                  const int rem = Kd - (kb + j) * 32;
                  const int ksteps = rem >= 32 ? 4 : (rem + 7) >> 3;   // 8 k-values per tf32 MMA; the padding is zero on both sides
                  for (int k = 0; k < ksteps; ++k) {
                    pc_mma(tacc, Ap + (uint64_t)(j * (kPcSlab >> 4) + k * 2), Bp + (uint64_t)(j * bstep + k * 2), idesc, acc);
                    acc = 1;
                  }
                }
                if (pass == 0) pc_commit(&lo_empty[l.slot]);
              }
            }
            pc_commit(&raw_empty[r.slot]);  // stage reusable once these MMAs have read it
          }
          __syncwarp();
          acc = 1;
          r.next(S), l.next(LS);
        }
      }
      if (pc_elect_one()) pc_commit(&tfull[a]);         // accumulators complete
      __syncwarp();
    }
  } else if (warp < kPcFirstEpi) {
    // ===================================================== split: lo = rn_tf32(x - trunc_tf32(x)), same (swizzled) offsets
    const int t = tid - kPcFirstSplit * 32;  // 0..63
    constexpr int kSplitThreads = kPcSplitWarps * 32;
    constexpr int kBatch = (int)(kPcSlab / 16u) / kSplitThreads;     // 16 float4 per thread per slab
    const int ngroups = (KB + G - 1) / G;
    PcRing r, l;
    for (int64_t u = 0; u < my_tiles * p.nsrc; ++u) {
      for (int gi = 0; gi < ngroups; ++gi) {
        const int ns = KB - gi * G < G ? KB - gi * G : G;
        pc_mbar_wait(&raw_full[r.slot], r.phase);
        const float4* __restrict__ src = reinterpret_cast<const float4*>(As + (size_t)r.slot * kStage);
        float4* __restrict__ dst = reinterpret_cast<float4*>(Ls + (size_t)l.slot * kStage);
        float4 x[kBatch];
#pragma unroll
        for (int j = 0; j < kBatch; ++j) x[j] = src[j * kSplitThreads + t];
        pc_mbar_wait(&lo_empty[l.slot], l.phase ^ 1u);
        for (int b = 0; b < ns; ++b) {
#pragma unroll
          for (int j = 0; j < kBatch; ++j)
            dst[(b * kBatch + j) * kSplitThreads + t] = make_float4(pc_lo(x[j].x), pc_lo(x[j].y), pc_lo(x[j].z), pc_lo(x[j].w));
          if (b + 1 < ns) {
#pragma unroll
            for (int j = 0; j < kBatch; ++j) x[j] = src[((b + 1) * kBatch + j) * kSplitThreads + t];
          }
        }
        pc_proxy_fence();
        pc_mbar_arrive(&lo_full[l.slot]);
        r.next(S), l.next(LS);
      }
    }
  } else {
    // ===================================================== epilogue: 8 warps = 4 TMEM lane quarters x 2 column halves
    const int ew = warp - kPcFirstEpi;
    const int quarter = warp & 3, half = ew >> 2;   // a warp may only touch TMEM lanes 32*(warp%4)..+31
    uint8_t* Et = Es + ew * 4096;
    uint64_t keep_policy;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep_policy));
    const int lrow = lane >> 3, lchunk = lane & 7;   // coalesced phase: 4 rows x 8 chunks of 16 bytes per pass
    constexpr int NGA = NG > 0 ? NG : 1;
    int ix[NGA][8], ixn[NGA][8];
    float cf[NGA][8], cfn[NGA][8];
    float rsc[2], rscn[2];
    auto load_ix = [&](int64_t tile_, int (&ixx)[NGA][8]) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t row = tile_ * kPcTileM + quarter * 32 + i * 4 + lrow;
#pragma unroll
        for (int g = 0; g < NGA; ++g) ixx[g][i] = (g < NG && row < p.M) ? __ldg(p.tidx[g] + row) : -1;
      }
    };
    auto load_cf = [&](int64_t tile_, float (&cff)[NGA][8], float (&rss)[2]) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t row = tile_ * kPcTileM + quarter * 32 + i * 4 + lrow;
#pragma unroll
        for (int g = 0; g < NGA; ++g) cff[g][i] = (g < NG && row < p.M) ? __ldg(p.tcoef[g] + row) : 0.f;
      }
      const int64_t myrow = tile_ * kPcTileM + quarter * 32 + lane;   // TMEM phase: lane = row
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const float* __restrict__ rsv = s ? p.rs[1] : p.rs[0];
        rss[s] = (s < p.nsrc && rsv && myrow < p.M) ? __ldg(rsv + myrow) : 1.f;
      }
    };
    auto load_idx = [&](int64_t tile_, int (&ixx)[NGA][8], float (&cff)[NGA][8], float (&rss)[2]) {
      load_ix(tile_, ixx);
      load_cf(tile_, cff, rss);
    };
    // row stride of the gathered tables and of `out`; a variable of its own because the lambdas capture it: writing Nd in its
    // place changes the register allocation of the three non-PSUM instantiations
    const int Tld = Nd;
    auto gather = [&](const int (&ixx)[NGA][8], int c0_, float4 (&g4)[NGA][8]) {
      const int lcol_ = c0_ + lchunk * 4, col_ = n0 + lcol_;
      const bool ok = lcol_ < Nsub && col_ < Nd;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int g = 0; g < NGA; ++g) {
          g4[g][i] = (NG > g && ixx[g][i] >= 0 && ok)
                         ? pc_ldg_keep(reinterpret_cast<const float4*>(p.T[g] + (size_t)ixx[g][i] * Tld + col_), keep_policy) : f4_zero();
        }
      }
    };
    float4 gv[NGA][8];
    if (grp < ntiles) load_idx(grp, ix, cf, rsc);
    for (int64_t ti = 0; ti < my_tiles; ++ti) {
      const int64_t tile = grp + ti * ngrp;
      const int a = (int)(ti & 1);
      const uint32_t taddr = tmem_base + (uint32_t)(a * (p.tmem_cols >> 1)) + ((uint32_t)(quarter * 32) << 16);
      const int64_t wrow0 = tile * kPcTileM + quarter * 32;
      bool waited = false;
      for (int c0 = half * 32; c0 < Nsub; c0 += 64) {
        const int lcol = c0 + lchunk * 4;        // column inside this CTA's window
        const int col = n0 + lcol;               // column of `out`
        const bool cok = lcol < Nsub && col < Nd;
        // gathered rows first: they do not depend on the accumulator, so their latency hides behind the wait for it
        gather(ix, c0, gv);
        if (!waited) {
          // next tile's indices / coefficients / row scales - one more load latency off the chain (NG <= 1: registers)
          if (NG <= 1 && ti + 1 < my_tiles) load_idx(tile + ngrp, ixn, cfn, rscn);
          pc_mbar_wait(&tfull[a], (uint32_t)((ti >> 1) & 1));
          pc_fence_after();
          waited = true;
        }
        // TMEM -> registers (lane = row), row scale and source sum, transpose through smem: 16-byte chunk q of row
        // `lane` goes to chunk q ^ (lane & 7)
#pragma unroll
        for (int q2 = 0; q2 < 4; ++q2) {
          uint32_t v0[8], v1[8];
          pc_tmem_ld8(taddr + c0 + q2 * 8, v0);
          if (p.nsrc > 1) pc_tmem_ld8(taddr + Nsp + c0 + q2 * 8, v1);
          pc_tmem_wait_ld();
          if constexpr (APAIR) {
#pragma unroll
            for (int e = 0; e < 8; ++e) v0[e] = __shfl_sync(0xffffffffu, v0[e], lane >> 1);
          }
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = rsc[0] * __uint_as_float(v0[e]);
          if (p.nsrc > 1) {
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = fmaf(rsc[1], __uint_as_float(v1[e]), o[e]);
          }
          *reinterpret_cast<float4*>(Et + lane * 128 + (((q2 * 2) ^ (lane & 7)) << 4)) = make_float4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<float4*>(Et + lane * 128 + (((q2 * 2 + 1) ^ (lane & 7)) << 4)) = make_float4(o[4], o[5], o[6], o[7]);
        }
        __syncwarp();
        float4 bsum = f4_zero(), bsq = f4_zero();
        const float4 bias4 = (p.bias && cok) ? __ldg(reinterpret_cast<const float4*>(p.bias + col)) : f4_zero();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rl = i * 4 + lrow;
          const int64_t row = wrow0 + rl;
          float4 o = *reinterpret_cast<const float4*>(Et + rl * 128 + ((lchunk ^ (rl & 7)) << 4));
          const bool live = row < p.M && cok;
          if (live) {
#pragma unroll
            for (int g = 0; g < NGA; ++g)
              if (NG > g) f4_fma(o, cf[g][i], gv[g][i]);
            f4_add(o, bias4);
          }
          if constexpr (PSUM) {
            // rows 2k / 2k+1 (the two directions of one pair) sit in lanes l and l ^ 8 (lrow = lane >> 3): the consumer - the
            // pair-init backward - only ever wants their SUM, so one row per pair is written (half the bytes here, half the
            // bytes of both of its passes). Whole-warp shuffles outside the `live` branch; M is even, so mates live together.
            float4 m;
            m.x = __shfl_xor_sync(0xffffffffu, o.x, 8), m.y = __shfl_xor_sync(0xffffffffu, o.y, 8);
            m.z = __shfl_xor_sync(0xffffffffu, o.z, 8), m.w = __shfl_xor_sync(0xffffffffu, o.w, 8);
            if (live && !(lrow & 1)) {
              f4_add(o, m);
              __stcs(reinterpret_cast<float4*>(p.out + (row >> 1) * Tld + col), o);
            }
          } else if (live) {
            // written once, read by a later kernel: evict first
            __stcs(reinterpret_cast<float4*>(p.out + row * Tld + col), o);
            f4_add(bsum, o);
            bsq.x = fmaf(o.x, o.x, bsq.x), bsq.y = fmaf(o.y, o.y, bsq.y), bsq.z = fmaf(o.z, o.z, bsq.z), bsq.w = fmaf(o.w, o.w, bsq.w);
          }
        }
        if (p.stats_part) {
          // lanes with the same chunk (lane & 7) hold partial sums of the same 4 columns: fixed-order xor tree,
          // then one lane per chunk adds the 32-row partial to this warp's double accumulators in smem
          float ps[8] = {bsum.x, bsum.y, bsum.z, bsum.w, bsq.x, bsq.y, bsq.z, bsq.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            ps[e] += __shfl_xor_sync(0xffffffffu, ps[e], 8);
            ps[e] += __shfl_xor_sync(0xffffffffu, ps[e], 16);
          }
          if (lrow == 0 && lcol < Nsub) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              red[(ew * 2 + 0) * Nsub + lcol + e] += (double)ps[e];
              red[(ew * 2 + 1) * Nsub + lcol + e] += (double)ps[4 + e];
            }
          }
        }
        __syncwarp();
      }
      if (!waited) {  // this warp has no column block (Nsub <= 32 and half == 1): still take part in the handshake
        if (NG <= 1 && ti + 1 < my_tiles) load_idx(tile + ngrp, ixn, cfn, rscn);
        pc_mbar_wait(&tfull[a], (uint32_t)((ti >> 1) & 1));
        pc_fence_after();
      }
      pc_fence_before();
      pc_mbar_arrive(&tempty[a]);
      if (NG <= 1) {
#pragma unroll
        for (int i = 0; i < 8; ++i) ix[0][i] = ixn[0][i], cf[0][i] = cfn[0][i];
        rsc[0] = rscn[0], rsc[1] = rscn[1];
      } else if (ti + 1 < my_tiles) {
        load_idx(tile + ngrp, ix, cf, rsc);
      }
    }
  }
  pc_fence_before();
  __syncthreads();
  if (p.stats_part) {
    for (int i = tid; i < 2 * Nsub; i += kPcThreads) {
      const int v = i / Nsub, c = i % Nsub;
      double s = 0;
      for (int w = 0; w < kPcEpilogueWarps; ++w) s += red[(w * 2 + v) * Nsub + c];
      p.stats_part[((size_t)blockIdx.x * 2 + v) * Nsub + c] = s;
    }
  }
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
}

// mean / inv_std of GraphNorm from per-CTA (sum, sum of squares) double partials (norm.cu semantics); CTA b holds the
// columns of window b % nsplit
__global__ void k_pc_stats_final(const double* __restrict__ part, int nparts, int nsplit, int Nsub, int64_t M, int C,
                                 const float* __restrict__ mean_scale, float eps, float* __restrict__ stats,
                                 double* __restrict__ moments) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const int split = c / Nsub, cl = c % Nsub;
  double s = 0, q = 0;
  for (int b = split; b < nparts; b += nsplit) {
    s += part[((size_t)b * 2 + 0) * Nsub + cl];
    q += part[((size_t)b * 2 + 1) * Nsub + cl];
  }
  if (moments) moments[c] = s, moments[C + c] = q;  // raw column sums for a row-sharded caller (summed over ranks, then
                                                    // twowl_graphnorm_stats_from_moments)
  const double mean = s / (double)M;
  double var = q / (double)M - mean * mean;
  if (var < 0) var = 0;
  const double a = (double)mean_scale[c];
  stats[c] = (float)mean;
  stats[C + c] = (float)(1.0 / sqrt(var + (1.0 - a) * (1.0 - a) * mean * mean + (double)eps));
}

// How one launch is cut: column windows of Nsub (multiple of 16) output columns per CTA, raw / lo ring depths.
struct PcConfig {
  int nsplit = 0, Nsub = 0, stages = 0, lo_stages = 0, tmem_cols = 0, group = kPcGroup;
  size_t smem = 0;
};
static size_t pc_smem_bytes(int Kd, int Nsub, int nsrc, bool with_stats, int stages, int lo_stages, int group) {
  const int KB = (Kd + 31) / 32;
  return (size_t)nsrc * 2 * KB * Nsub * 128 + (size_t)(stages + lo_stages) * ((Kd + 31) / 32 > 1 ? group * kPcSlab : kPcSlab) + kPcEpilogueWarps * 4096 +
         (2 * kPcMaxStages + 2 * kPcMaxLo + 8) * 8 + (with_stats ? (size_t)kPcEpilogueWarps * 2 * Nsub * 8 : 0) + 1024;
}
static int pc_tmem_cols(int Nsub, int nsrc) {
  const int need = 2 * nsrc * ((Nsub + 31) / 32 * 32);   // the epilogue reads 32-column blocks
  int cols = 32;
  while (cols < need) cols <<= 1;
  return cols;
}
// Fewest column windows that fit at all: every extra window re-reads (and re-splits) the whole A tile, which costs far more than
// a shallower ring (measured at C = 128, M = 15 M: 2 windows with 2 raw stages 5.3 ms, 4 windows with 3 stages 8.2 ms, 8 windows
// 15.2 ms). The ring is then grown to what the remaining shared memory holds.
static PcConfig pc_config(int Kd, int Nd, int nsrc, bool with_stats) {
  PcConfig best;
  if (Kd < 4 || Kd > 1024 || (Kd % 4) || Nd < 4 || Nd > 1024 || (Nd % 4) || nsrc < 1 || nsrc > 2) return best;
  const size_t cap = 227 * 1024;
  for (int ns = 1; ns <= 32 && !best.nsplit; ns *= 2) {
    const int Nsub = (int)(cdiv(cdiv(Nd, ns), 16) * 16);
    if (Nsub > 256 || (ns > 1 && (int64_t)(ns - 1) * Nsub >= Nd)) continue;
    if (pc_tmem_cols(Nsub, nsrc) > 512) continue;
    int lo = 1, grp = kPcGroup, st = 2;
    if (pc_smem_bytes(Kd, Nsub, nsrc, with_stats, 2, lo, kPcGroup) > cap) {
      // two 32 KB stages do not fit: a ring of >= 3 single-slab (16 KB) stages still beats doubling the windows
      grp = 1, st = 3;
      if (pc_smem_bytes(Kd, Nsub, nsrc, with_stats, st, lo, grp) > cap) continue;
    }
    while (st < kPcMaxStages && pc_smem_bytes(Kd, Nsub, nsrc, with_stats, st + 1, lo, grp) <= cap) ++st;
    best.nsplit = ns, best.Nsub = Nsub, best.stages = st, best.lo_stages = lo, best.group = grp;
    best.tmem_cols = pc_tmem_cols(Nsub, nsrc);
    best.smem = pc_smem_bytes(Kd, Nsub, nsrc, with_stats, st, lo, grp);
  }
  return best;
}
static bool pc_supported(int Kd, int Nd, int nsrc) { return pc_config(Kd, Nd, nsrc, nsrc == 1).nsplit > 0; }
static int pc_grid(int64_t M, int nsplit) {
  const int64_t ntiles = cdiv(M, kPcTileM);
  const int64_t groups = kNumSMs / nsplit;
  return (int)((ntiles < groups ? ntiles : groups) * nsplit);
}

// row-major fp32 [M, Kd] -> boxes of 32 columns x 128 rows, SWIZZLE_128B (the UMMA K-major canonical layout); columns
// beyond Kd are zero-filled by the TMA unit
static int pc_make_tmap(CUtensorMap* tm, const float* A, int64_t M, int Kd) {
  return make_tmap_2d_f32(tm, A, M, Kd, 32, kPcTileM, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int NG, bool PSUM = false, bool APAIR = false>
static int pc_launch(const ConvParams& p, size_t smem, const CUtensorMap& t0, const CUtensorMap& t1, cudaStream_t s) {
  TW_CUDA(cudaFuncSetAttribute(k_pair_conv<NG, PSUM, APAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_pair_conv<NG, PSUM, APAIR><<<pc_grid(p.M, p.nsplit), kPcThreads, smem, s>>>(p, t0, t1);
  TW_LAUNCH_CHECK();
  return 0;
}

}  // namespace twowl

using namespace twowl;

extern "C" size_t twowl_sizeof_conv_args(void) { return sizeof(twowl_conv_args); }

extern "C" int twowl_pair_conv(const twowl_conv_args* a, void* ws, size_t ws_bytes, void* stream);

// The plain linear layer (linear.cu: twowl_linear_fwd / twowl_linear_bwd_input, impl 1 / 2) is this kernel with one
// source and no epilogue terms: C[M,Nd] = A[M,Kd] * B^T, B = W[Nd,Kd] (w_kn = 0) or W[Kd,Nd] (w_kn = 1).
namespace twowl {
bool linear_tc_supported(int Kd, int Nd) { return pc_config(Kd, Nd, 1, false).nsplit > 0; }
int linear_tc(const float* A, const float* W, float* C, int64_t M, int Kd, int Nd, int w_kn, cudaStream_t s) {
  twowl_conv_args a;
  memset(&a, 0, sizeof(a));
  a.nsrc = 1, a.Kd = Kd, a.Nd = Nd, a.M = M;
  a.A[0] = A, a.W[0] = W, a.w_kn[0] = w_kn, a.out = C;
  return twowl_pair_conv(&a, nullptr, 0, (void*)s);
}
}  // namespace twowl

extern "C" int twowl_pair_conv_supported(int32_t Kd, int32_t Nd, int32_t nsrc) { return pc_supported(Kd, Nd, nsrc) ? 1 : 0; }

extern "C" size_t twowl_pair_conv_workspace_bytes(int64_t M, int32_t Nd) {
  (void)M;
  return align_up((size_t)kNumSMs * 2 * (size_t)(Nd < 256 ? 256 : Nd) * sizeof(double));
}

extern "C" int twowl_pair_conv(const twowl_conv_args* a, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(a != nullptr && a->nsrc >= 1 && a->nsrc <= 2 && a->ngather >= 0 && a->ngather <= 2, "pair_conv: bad nsrc/ngather");
  TW_CHECK_ARG(a->M >= 0, "pair_conv: negative M");
  const bool want_stats = a->stats != nullptr;
  const PcConfig cfg = pc_config(a->Kd, a->Nd, a->nsrc, want_stats);
  TW_CHECK_ARG(cfg.nsplit > 0, "pair_conv: Kd=%d Nd=%d nsrc=%d%s unsupported (widths %% 4, <= 1024, shared memory)", a->Kd, a->Nd,
               a->nsrc, want_stats ? " with statistics" : "");
  ConvParams p;
  memset(&p, 0, sizeof(p));
  for (int s = 0; s < a->nsrc; ++s) {
    TW_CHECK_ARG(aligned16(a->A[s]) && aligned16(a->W[s]), "pair_conv: A/W must be 16-byte aligned");
    p.rs[s] = a->row_scale[s], p.W[s] = a->W[s], p.w_kn[s] = a->w_kn[s];
  }
  for (int g = 0; g < a->ngather; ++g) {
    TW_CHECK_ARG(a->T[g] && a->tidx[g] && a->tcoef[g] && aligned16(a->T[g]), "pair_conv: incomplete gather term %d", g);
    p.T[g] = a->T[g], p.tidx[g] = a->tidx[g], p.tcoef[g] = a->tcoef[g];
  }
  TW_CHECK_ARG(aligned16(a->out) && aligned16(a->bias), "pair_conv: out/bias must be 16-byte aligned");
  if (a->pair_sum_out) {
    TW_CHECK_ARG(!want_stats && a->M % 2 == 0 && a->ngather == 2,
                 "pair_conv: pair_sum_out is built for the pair layer's input gradient: two gathers, an even M, no statistics");
  }
  TW_CHECK_ARG(a->a_pairs == 0 || a->a_pairs == 1, "pair_conv: a_pairs = %d (0 or 1)", a->a_pairs);
  if (a->a_pairs) {
    TW_CHECK_ARG(a->nsrc == 1 && a->ngather == 1 && a->M % 2 == 0 && !a->pair_sum_out,
                 "pair_conv: a_pairs is built for the depth-1 pair layer's forward: one source, one gather, an even M");
  }
  p.nsrc = a->nsrc, p.ngather = a->ngather, p.M = a->M, p.Kd = a->Kd, p.Nd = a->Nd, p.bias = a->bias, p.out = a->out;
  p.Nsub = cfg.Nsub, p.nsplit = cfg.nsplit, p.stages = cfg.stages, p.lo_stages = cfg.lo_stages, p.tmem_cols = cfg.tmem_cols, p.group = cfg.group;
  cudaStream_t s = (cudaStream_t)stream;
  if (want_stats) {
    TW_CHECK_ARG(a->mean_scale != nullptr && a->M > 0, "pair_conv: stats need mean_scale and M > 0");
    TW_CHECK_WS(ws_bytes, twowl_pair_conv_workspace_bytes(a->M, a->Nd));
    p.stats_part = (double*)ws;
  }
  if (a->M == 0) return 0;
  CUtensorMap tm[2];
  memset(tm, 0, sizeof(tm));
  for (int i = 0; i < a->nsrc; ++i) {
    // a_pairs: A has one row per pair, fetched as 16-row boxes (four per 128-row output tile)
    const int rc_t = a->a_pairs ? make_tmap_2d_f32(&tm[i], a->A[i], a->M / 2, a->Kd, 32, 16, CU_TENSOR_MAP_SWIZZLE_128B)
                                : pc_make_tmap(&tm[i], a->A[i], a->M, a->Kd);
    if (rc_t) return rc_t;
  }
  const int rc = a->a_pairs        ? pc_launch<1, false, true>(p, cfg.smem, tm[0], tm[1], s)
                 : a->pair_sum_out ? pc_launch<2, true>(p, cfg.smem, tm[0], tm[1], s)
                 : a->ngather == 0 ? pc_launch<0>(p, cfg.smem, tm[0], tm[1], s)
                 : a->ngather == 1 ? pc_launch<1>(p, cfg.smem, tm[0], tm[1], s)
                                   : pc_launch<2>(p, cfg.smem, tm[0], tm[1], s);
  if (rc) return rc;
  if (want_stats) {
    k_pc_stats_final<<<(int)cdiv(a->Nd, 128), 128, 0, s>>>(p.stats_part, pc_grid(a->M, cfg.nsplit), cfg.nsplit, cfg.Nsub, a->M, a->Nd,
                                                           a->mean_scale, a->eps, a->stats, a->moments);
    TW_LAUNCH_CHECK();
  }
  return 0;
}
