// dw_tc.cu - weight gradients of the two pair-level linear layers in ONE pass on tcgen05 tensor cores:
//
//   [dW_f ; dW_r] (2C x C)  =  [ selfw_f * dO_f | selfw_r * dO_r ]^T (2C x M)  *  H (M x C)
//
// (reference: autograd of GCNConv.lin at TwoWL/model/model.py:37 for conv2s[i] and conv2s_r[i], which share
// their input H - model.py:77). The reduction runs over M = rows of the pair table, so both operands are used
// in their natural row-major form as MN-MAJOR UMMA operands: a 64-row tile of dO_f/dO_r is the A operand [128 x 64k],
// the same rows of H are the B operand [C x 64k]; tcgen05.mma kind::tf32, 3xTF32 split. H is read once for both
// directions: 3 reads of [M,C] in total.
//
// One persistent CTA per SM, 14 warps, warp-specialised:
//   warp  0    TMA producer: raw fp32 tiles of dO_f, dO_r, H with cp.async.bulk.tensor (SWIZZLE_128B_ATOM_32B tensor maps
//                            = the one MN-major layout the tensor core accepts for tf32, see below), L2 evict-first
//   warps 2-9  split       : A: v = selfw[row] * raw written back in place (the tensor core truncates it to tf32 = the `hi`
//                            operand) and lo = v - trunc(v) into a second buffer; B: lo only (raw H is its own hi)
//   warp  1    MMA issuer  : 3 x 8 tcgen05.mma per tile into a TMEM accumulator that is drained every kDwFlush tiles
//   warps 10-13 drain      : TMEM -> fp32 registers after every tile (C <= 64), 64 tiles per addition into the CTA's double
//                            partials in global memory; a second kernel adds the partials in double in CTA order:
//                            deterministic.
#include "common.cuh"

#ifndef TWOWL_DW_FLUSH
#define TWOWL_DW_FLUSH 2
#endif

namespace twowl {

constexpr int kDwSplitWarps = 8;    // the split pass is latency-bound per warp: 8 warps halve each thread's rows
constexpr int kDwFirstSplit = 2;
constexpr int kDwFirstDrain = kDwFirstSplit + kDwSplitWarps;   // 10
constexpr int kDwThreads = (kDwFirstDrain + 4) * 32;           // 448
constexpr int kDwStages = 2;
// per width C: rows of the pair table per stage (the stage holds hi + lo of dO_f, dO_r and H: 96 KB at C = 64 / TK = 64 and at
// C = 128 / TK = 32), accumulators (C <= 64: ONE 128-row D = [f cols | r cols]; C = 128: D_f and D_r), tiles accumulated in
// TMEM between drains (1024 rows)
__host__ __device__ constexpr int dw_tile_k(int C) { return C <= 64 ? 64 : 32; }
__host__ __device__ constexpr int dw_nacc(int C) { return C <= 64 ? 1 : 2; }
// The tensor core's fp32 accumulate TRUNCATES: a TMEM-resident sum loses about half an ulp of its own magnitude per
// accumulate step, always towards zero (2048 rows at C = 128 measured 1.6e-5 relative in round 1, when both widths drained
// after 384 steps - above the 1e-5 band of a weight gradient). C <= 64 therefore drains every TWOWL_DW_FLUSH = 2 tiles (the
// first tile's small products are added while the accumulator is still small: ~32 steps at full magnitude, < 2e-6
// relative; every tile: 0.5 ms slower for 5e-7); the drain warps add the drains in fp32 registers, 64 at a time, into
// per-CTA DOUBLE partials. C = 128 (two 128 x 128 accumulators, no room in registers: the running sums live in `part`, a
// 128 KB read-add-write per drain) drains every 8 tiles of 32 rows: ~96 steps, < 6e-6 relative (every 4 tiles was measured:
// the read-add-write traffic made the kernel 1.7x slower at R = 60 M).
__host__ __device__ constexpr int dw_flush(int C) { return C <= 64 ? TWOWL_DW_FLUSH : 8; }
constexpr int kDwRegTiles = 64;   // C <= 64: tiles added in fp32 registers between two additions into the double partials
__host__ __device__ constexpr int dw_part_rows(int C) { return C <= 64 ? 128 : 2 * C; }

struct DwParams {
  const float* rsf;
  const float* rsr;
  int64_t M;
  float* part;  // [gridDim.x][dw_part_rows(C)][C]: fp32 running sums (C = 128), or the same shape in double (C <= 64)
  // GN = true: the A tiles are the OUTPUTS O_f, O_r of the last pair layer and the gradients are made on the fly
  // (twowl_pair_dw_gn): dO = P * O + Q (+ sc * g_y on the rows the readout selected), written to dOf / dOr as well
  const float* consts;   // [2 branches][4][C] = (P, Q, sc, of), twowl_gn2_readout_bwd_finish
  const float* G;        // [2L, C] gradient of the selected rows, by position
  const int32_t* head;   // [M] first position that selects a row, -1 = none
  const int32_t* next;   // [2L] next position selecting the same row
  float* dOf;
  float* dOr;
  uint32_t thresh;
  float inv_keep;
  uint64_t seed_f, seed_r;
  int relu;
};

__device__ __forceinline__ uint32_t dw_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// MN-major tf32 operands: on sm_100a the tensor core accepts ONLY layout type 1 (SWIZZLE_128B_BASE32B) for a transposed
// tf32 operand - every other layout type makes tcgen05.mma write zeros (measured with tools/mma_probe.cu). The layout,
// as the hardware reads it (same probe): element (mn, k) of an operand lives at byte
//   (mn / 32) * LBO + (k / 4) * SBO + (k % 4) * 128 + ((((mn % 32) / 8) ^ (k % 4)) * 32) + (mn % 8) * 4
// i.e. 512-byte atoms of 4 k-rows x 32 mn-elements whose 32-byte units are XOR-swizzled by the k-row (Swizzle<2,5,2>).
// With SBO = 512 a group of 32 mn-elements is [64 k-rows][128 B] - exactly what a TMA box of 32 columns x 64 rows with
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B writes, so row-major global tiles land in operand layout without a register pass.
constexpr uint32_t kDwSbo = 512u;                                   // next group of 4 k-rows
constexpr uint32_t kDwKStep = 2u * kDwSbo;                          // one tf32 MMA consumes 8 k-rows
__device__ __forceinline__ uint64_t dw_desc(uint32_t saddr, uint32_t lbo) {   // lbo: next group of 32 mn-elements
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((kDwSbo >> 4) & 0x3FFFu) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}
__device__ __forceinline__ void dw_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(dw_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void dw_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(dw_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void dw_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(dw_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void dw_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dw_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void dw_tma_load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
          dw_smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(dw_smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void dw_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(dw_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void dw_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void dw_tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// one lane of a converged warp: the loops around the single-thread instructions run on the whole warp with warp-uniform
// values, so descriptors live in uniform registers and the UTCHMMA / UTMALDG issue back to back (see pair_conv.cu)
__device__ __forceinline__ bool dw_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// tf32 split (see pair_conv.cu): the tensor core reads an fp32 operand as hi = trunc_tf32(x); lo = x - hi goes into a second
// buffer for both operands, three products. (Rounding hi / lo to nearest as pair_conv does for its lo was measured here: the
// extra integer work sits on the split warps' critical path - +1.0 ms of 15 - for no change of any end-to-end error.)
__device__ __forceinline__ float dw_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

// C = width of dO_f, dO_r and H (32, 64 or 128). One stage:
//   A_hi: AG groups of 32 M-elements ([f cols | r cols | zero padding when C = 32]), A_lo: the same, B_hi: C/32 groups, B_lo
// HP (H at half height, twowl_pair_dw_gn with h_pairs = 1): H holds ONE row per pair, H[k] = rows 2k and 2k+1 of the pair
// table. TMA lands the tile's TK/2 rows in a staging area (Hs, C/32 groups of TK/2 rows) and the split warps write each of them
// twice, to K-rows 2k and 2k+1 of B_hi (raw) and B_lo (split): the MMAs see the same operands in the same K order as with the
// full-height H, so the sums are bit-identical (adding mates before the MMA would halve its work but change the rounding).
template <int C, bool GN, bool HP = false>
__global__ void __launch_bounds__(kDwThreads, 1) k_dw_tc(const DwParams p, const __grid_constant__ CUtensorMap tmF,
                                                         const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmH) {
  constexpr int GS = C / 32;                          // 32-column groups per source
  constexpr int kDwTileK = dw_tile_k(C), NACC = dw_nacc(C), kDwFlush = dw_flush(C);
  constexpr int AG = NACC == 1 ? 4 : 2 * GS;          // A groups: one 128-row D (C <= 64) or D_f | D_r of 128 rows each
  constexpr int TB = NACC == 1 ? 64 : 2 * C;          // TMEM columns per accumulator buffer
  constexpr uint32_t kDwLbo = (kDwTileK / 4) * kDwSbo;   // next group of 32 mn-elements
  constexpr uint32_t kAHalf = (uint32_t)AG * kDwLbo;  // hi (or lo) part of the A stage
  constexpr uint32_t kBHalf = (uint32_t)GS * kDwLbo;
  constexpr uint32_t kHs = HP ? (uint32_t)GS * (kDwLbo / 2) : 0u;   // staging of the half-height H tile
  constexpr uint32_t kStage = 2u * kAHalf + 2u * kBHalf + kHs;
  constexpr uint32_t kTxBytes = 2u * GS * kDwLbo + (HP ? kHs : (uint32_t)GS * kDwLbo);   // raw bytes landing per tile
  extern __shared__ uint8_t dw_smem_raw[];
  // 1024-byte alignment by OFFSET from the shared array: a pointer rebuilt from an integer would be generic (LD.E / ST.E)
  uint8_t* smem = dw_smem_raw + ((1024u - (dw_smem_u32(dw_smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kDwStages * kStage);
  uint64_t* raw_full = bars;        // [stages] TMA -> split
  uint64_t* split_done = bars + 2;  // [stages] split -> MMA
  uint64_t* empty = bars + 4;       // [stages] MMA -> TMA
  uint64_t* tfull = bars + 6;       // [2] MMA -> drain
  uint64_t* tempty = bars + 8;      // [2] drain -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);
  float* cs = reinterpret_cast<float*>(bars + 16);   // GN: [2 branches][P, Q][C] column constants

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // dropout seeds as VALUES, read once: a tagged seed is the address of a device uint64 (common.cuh). Resolving inside the split
  // pass - a load the compiler must keep ordered against that pass's stores - cost 3.4 ms of the 14.6 (measured).
  uint64_t seed_f = 0, seed_r = 0;
  if (GN && p.thresh) seed_f = resolve_seed(p.seed_f), seed_r = resolve_seed(p.seed_r);
  const int64_t ntiles = (p.M + kDwTileK - 1) / kDwTileK;
  const int64_t my_tiles = (ntiles > blockIdx.x) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dw_smem_u32(tmem_slot)), "r"(2 * TB) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int s = 0; s < kDwStages; ++s) {
      dw_mbar_init(&raw_full[s], 1);
      dw_mbar_init(&split_done[s], kDwSplitWarps * 32);
      dw_mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      dw_mbar_init(&tfull[a], 1);
      dw_mbar_init(&tempty[a], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmF)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmR)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmH)) : "memory");
  }
  if (GN)
    for (int i = tid; i < 4 * C; i += kDwThreads) cs[i] = __ldg(p.consts + (i / (2 * C)) * 4 * C + (i % (2 * C)));
  // zero the padding groups of A (C = 32 only): written once, never touched again
  if (2 * GS < AG) {
    for (int st = 0; st < kDwStages; ++st)
      for (int half = 0; half < 2; ++half) {
        float4* z = reinterpret_cast<float4*>(smem + st * kStage + half * kAHalf + 2 * GS * kDwLbo);
        for (int i = tid; i < (int)((AG - 2 * GS) * kDwLbo / 16); i += kDwThreads) z[i] = f4_zero();
      }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // provably warp-uniform

  if (warp == 0) {
    // ===================================================== TMA producer
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t tile = blockIdx.x + it * gridDim.x;
      const int st = (int)(it % kDwStages);
      const int row = (int)(tile * kDwTileK);
      dw_mbar_wait(&empty[st], (uint32_t)(((it / kDwStages) & 1) ^ 1));
      if (dw_elect_one()) {
        dw_mbar_expect_tx(&raw_full[st], kTxBytes);
        uint8_t* Ahi = smem + st * kStage;
        uint8_t* Bhi = Ahi + 2 * kAHalf;
#pragma unroll
        for (int g = 0; g < GS; ++g) {
          dw_tma_load_2d(Ahi + (size_t)g * kDwLbo, &tmF, g * 32, row, &raw_full[st], policy);
          dw_tma_load_2d(Ahi + (size_t)(GS + g) * kDwLbo, &tmR, g * 32, row, &raw_full[st], policy);
          if (HP)
            dw_tma_load_2d(Bhi + 2 * kBHalf + (size_t)g * (kDwLbo / 2), &tmH, g * 32, row / 2, &raw_full[st], policy);
          else
            dw_tma_load_2d(Bhi + (size_t)g * kDwLbo, &tmH, g * 32, row, &raw_full[st], policy);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    // D[128, C] (+)= A[128 x 8] * B[C x 8]^T per K-step; A and B both MN-major
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t grp = it / kDwFlush;
      const int a = (int)(grp & 1);
      if (it % kDwFlush == 0) {
        dw_mbar_wait(&tempty[a], (uint32_t)(((grp >> 1) & 1) ^ 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      }
      const int st = (int)(it % kDwStages);
      dw_mbar_wait(&raw_full[st], (uint32_t)((it / kDwStages) & 1));
      dw_mbar_wait(&split_done[st], (uint32_t)((it / kDwStages) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // descriptors advance by byte offset >> 4 in their low word
      const uint64_t Ahi = dw_desc(dw_smem_u32(smem) + (uint32_t)st * kStage, kDwLbo);
      const uint64_t Alo = Ahi + (kAHalf >> 4), Bhi = Alo + (kAHalf >> 4), Blo = Bhi + (kBHalf >> 4);
      const uint32_t acc0 = (it % kDwFlush == 0) ? 0u : 1u;
      const bool last = (it + 1) % kDwFlush == 0 || it + 1 == my_tiles;
      if (dw_elect_one()) {
#pragma unroll
        for (int ac = 0; ac < NACC; ++ac) {   // C = 128: D_f from the f groups of A, D_r from the r groups
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {   // lo*hi, hi*lo, hi*hi: small terms first
            const uint64_t Ap = ((pass == 0) ? Alo : Ahi) + (uint64_t)(ac * GS * (kDwLbo >> 4));
            const uint64_t Bp = (pass == 1) ? Blo : Bhi;
#pragma unroll
            for (int k = 0; k < kDwTileK / 8; ++k)   // one group of 8 k-rows per K-step
              dw_mma(tmem_base + (uint32_t)(a * TB + ac * C), Ap + (uint64_t)(k * (kDwKStep >> 4)), Bp + (uint64_t)(k * (kDwKStep >> 4)),
                     idesc, (pass | k) ? 1u : acc0);
          }
        }
        dw_commit(&empty[st]);
        if (last) dw_commit(&tfull[a]);
      }
      __syncwarp();
    }
  } else if (warp < kDwFirstDrain) {
    // ===================================================== split (scale + hi/lo), linear over the swizzled buffers
    const int t = tid - kDwFirstSplit * 32;                  // 0..127
    constexpr int kSplitThreads = kDwSplitWarps * 32;
    constexpr int RPT = kDwTileK * 8 / kSplitThreads;        // pair-table rows per split thread (8 threads cover a row's 128 B)
    constexpr int RSTEP = kSplitThreads / 8;                 // rows between a thread's consecutive rows
    constexpr int kAChunks = 2 * GS * (int)(kDwLbo / 16);    // 16-byte chunks of the live A groups (f then r)
    constexpr int kBChunks = GS * (int)(kDwLbo / 16);
    constexpr int kBIter = kBChunks / kSplitThreads;
    static_assert(kAChunks == 2 * GS * RPT * kSplitThreads, "RPT rows x 2*GS chunks per split thread");
    // chunk i of a group region sits in k-row (i % 512) / 8; with i = j*kSplitThreads + t that is (j % RPT) * RSTEP + t / 8
    // GN: this thread's 4 columns inside a 32-column group are fixed (unit ((t & 7) >> 1) ^ (k & 3), k & 3 = (t >> 3) & 3), so
    // the per-column constants of its (branch, group) chunks are 2 LDS.128 per chunk
    const int tcol = (((((t & 7) >> 1) ^ ((t >> 3) & 3))) << 3) + ((t & 1) << 2);
    // Everything a tile needs from global memory besides the TMA data is loaded ONE tile ahead (row scales, chain links, the
    // selected rows' gradients) and the chain heads TWO tiles ahead (the gradients' addresses depend on them), so no global
    // load latency sits between the arrival of a tile and its transform.
    float sf[RPT], sr[RPT], sfn[RPT], srn[RPT];
    int hd[RPT], nx[RPT], hdn[RPT], nxn[RPT], hdnn[RPT];
    float4 Gd[RPT][GN ? GS : 1], Gdn[RPT][GN ? GS : 1];
    const int64_t tstride = (int64_t)gridDim.x * kDwTileK;
    auto load_heads = [&](int64_t row0_, bool live, int (&h)[RPT]) {
#pragma unroll
      for (int q = 0; q < RPT; ++q) {
        const int64_t row = row0_ + q * RSTEP + (t >> 3);
        h[q] = (GN && live && row < p.M) ? __ldg(p.head + row) : -1;
      }
    };
    auto load_rows = [&](int64_t row0_, bool live, const int (&h)[RPT], float (&a)[RPT], float (&b)[RPT], int (&n)[RPT], float4 (&g)[RPT][GN ? GS : 1]) {
#pragma unroll
      for (int q = 0; q < RPT; ++q) {
        const int64_t row = row0_ + q * RSTEP + (t >> 3);
        const bool ok = live && row < p.M;
        a[q] = ok ? __ldg(p.rsf + row) : 0.f;
        b[q] = ok ? __ldg(p.rsr + row) : 0.f;
        n[q] = -1;
        if (GN) {
          if (h[q] >= 0) n[q] = __ldg(p.next + h[q]);
#pragma unroll
          for (int gi = 0; gi < GS; ++gi)
            g[q][gi] = h[q] >= 0 ? ldg_cached(reinterpret_cast<const float4*>(p.G + (int64_t)h[q] * C + gi * 32 + tcol)) : f4_zero();
        }
      }
    };
    {
      const int64_t r0 = (int64_t)blockIdx.x * kDwTileK;
      load_heads(r0, my_tiles > 0, hdn);
      load_heads(r0 + tstride, my_tiles > 1, hdnn);
      load_rows(r0, my_tiles > 0, hdn, sfn, srn, nxn, Gdn);
    }
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t tile = blockIdx.x + it * gridDim.x;
      const int st = (int)(it % kDwStages);
      const int64_t row0 = tile * kDwTileK;
#pragma unroll
      for (int q = 0; q < RPT; ++q) {
        sf[q] = sfn[q], sr[q] = srn[q], hd[q] = hdn[q], nx[q] = nxn[q], hdn[q] = hdnn[q];
#pragma unroll
        for (int gi = 0; gi < (GN ? GS : 1); ++gi) Gd[q][gi] = Gdn[q][gi];
      }
      dw_mbar_wait(&raw_full[st], (uint32_t)((it / kDwStages) & 1));
      // next tile's row data and the heads of the tile after it: in flight while this tile is transformed
      load_rows(row0 + tstride, it + 1 < my_tiles, hdn, sfn, srn, nxn, Gdn);
      load_heads(row0 + 2 * tstride, it + 2 < my_tiles, hdnn);
      float4* Ahi = reinterpret_cast<float4*>(smem + st * kStage);
      float4* Alo = reinterpret_cast<float4*>(smem + st * kStage + kAHalf);
      const float4* Bhi = reinterpret_cast<const float4*>(smem + st * kStage + 2 * kAHalf);
      float4* Blo = reinterpret_cast<float4*>(smem + st * kStage + 2 * kAHalf + kBHalf);
      // one branch (f, then r) at a time: RPT rows x GS column groups per thread
#pragma unroll
      for (int br = 0; br < 2; ++br) {
        float4 v[GS][RPT];
        // phase 1, branch-free: load, dense part of the GraphNorm backward
#pragma unroll
        for (int gi = 0; gi < GS; ++gi) {
#pragma unroll
          for (int q = 0; q < RPT; ++q) {
            const int j = (br * GS + gi) * RPT + q;
            float4 x = Ahi[j * kSplitThreads + t];
            if (GN) {
              const float4 P4 = *reinterpret_cast<const float4*>(cs + br * 2 * C + gi * 32 + tcol);
              const float4 Q4 = *reinterpret_cast<const float4*>(cs + br * 2 * C + C + gi * 32 + tcol);
              x = make_float4(fmaf(P4.x, x.x, Q4.x), fmaf(P4.y, x.y, Q4.y), fmaf(P4.z, x.z, Q4.z), fmaf(P4.w, x.w, Q4.w));
            }
            v[gi][q] = x;
          }
        }
        // phase 2: rows the readout selected: + sc * (dropout / ReLU mask) * sum of their positions' gradients
        if (GN) {
#pragma unroll
          for (int q = 0; q < RPT; ++q) {
            if (hd[q] >= 0) {
              const int64_t row = row0 + q * RSTEP + (t >> 3);
#pragma unroll
              for (int gi = 0; gi < GS; ++gi) {
                const int col = gi * 32 + tcol;
                float4 d = Gd[q][gi];
                if (nx[q] >= 0) {   // selected more than once: positions in ascending order (deterministic)
                  const float4* __restrict__ G4 = reinterpret_cast<const float4*>(p.G + col);
                  d = f4_zero();
                  int last = -1;
                  for (;;) {
                    int best = 0x7fffffff;
                    for (int c = hd[q]; c >= 0; c = __ldg(p.next + c))
                      if (c > last && c < best) best = c;
                    if (best == 0x7fffffff) break;
                    f4_add(d, ldg_cached(G4 + (int64_t)best * (C / 4)));
                    last = best;
                  }
                }
                const float* __restrict__ cb = p.consts + (br ? 4 * C : 0) + col;
                const float4 S4 = __ldg(reinterpret_cast<const float4*>(cb + 2 * C)), O4 = __ldg(reinterpret_cast<const float4*>(cb + 3 * C));
                // the forward value y = sc*x + of from dO = P*x + Q would lose x when P is tiny: keep it exact from the raw tile
                const float4 xr = Ahi[((br * GS + gi) * RPT + q) * kSplitThreads + t];
                const float xa[4] = {xr.x, xr.y, xr.z, xr.w}, da[4] = {d.x, d.y, d.z, d.w}, sa[4] = {S4.x, S4.y, S4.z, S4.w},
                            oa[4] = {O4.x, O4.y, O4.z, O4.w};
                float add[4];
                const uint64_t e0 = (uint64_t)row * C + col;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                  float g = da[c], keep = 1.f;
                  if (p.thresh) keep = drop_scale(br ? seed_r : seed_f, e0 + c, p.thresh, p.inv_keep);
                  g *= keep;
                  if (p.relu && !(fmaf(sa[c], xa[c], oa[c]) * keep > 0.f)) g = 0.f;
                  add[c] = sa[c] * g;
                }
                v[gi][q].x += add[0], v[gi][q].y += add[1], v[gi][q].z += add[2], v[gi][q].w += add[3];
              }
            }
          }
        }
        // phase 3, branch-free: gradient out, row scale, hi (in place) / lo
#pragma unroll
        for (int gi = 0; gi < GS; ++gi) {
#pragma unroll
          for (int q = 0; q < RPT; ++q) {
            const int j = (br * GS + gi) * RPT + q;
            float4 x = v[gi][q];
            if (GN) {
              const int64_t row = row0 + q * RSTEP + (t >> 3);
              if (row < p.M) __stcs(reinterpret_cast<float4*>((br ? p.dOr : p.dOf) + row * C + gi * 32 + tcol), x);
            }
            const float sc = br ? sr[q] : sf[q];
            x.x *= sc, x.y *= sc, x.z *= sc, x.w *= sc;
            Ahi[j * kSplitThreads + t] = x;
            Alo[j * kSplitThreads + t] = make_float4(dw_lo(x.x), dw_lo(x.y), dw_lo(x.z), dw_lo(x.w));
          }
        }
      }
      if constexpr (HP) {
        // staging chunk i: group g, pair row k (byte k * 128 of the group), 32-byte unit us = logical unit u ^ (k & 3), half hh;
        // K-rows 2k and 2k+1 of B take it at their own swizzle phase
        constexpr int kHsGroupChunks = (int)(kDwLbo / 32);
        const float4* Hs = reinterpret_cast<const float4*>(smem + st * kStage + 2 * kAHalf + 2 * kBHalf);
        float4* Bh = reinterpret_cast<float4*>(smem + st * kStage + 2 * kAHalf);
#pragma unroll
        for (int j = 0; j < kBIter / 2; ++j) {
          const int i = j * kSplitThreads + t;
          const float4 v = Hs[i];
          const float4 lo = make_float4(dw_lo(v.x), dw_lo(v.y), dw_lo(v.z), dw_lo(v.w));
          const int g = i / kHsGroupChunks, o = i % kHsGroupChunks;   // o: 16-byte chunk inside the group's staging
          const int k = o >> 3, u = ((o >> 1) & 3) ^ (k & 3), hh = o & 1;
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int kk = 2 * k + e;
            const int c = g * (int)(kDwLbo / 16) + kk * 8 + ((u ^ (kk & 3)) << 1) + hh;
            Bh[c] = v;
            Blo[c] = lo;
          }
        }
      } else {
#pragma unroll 4
        for (int j = 0; j < kBIter; ++j) {
          const int i = j * kSplitThreads + t;
          const float4 v = Bhi[i];
          Blo[i] = make_float4(dw_lo(v.x), dw_lo(v.y), dw_lo(v.z), dw_lo(v.w));
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      dw_mbar_arrive(&split_done[st]);
    }
  } else {
    // ===================================================== drain: a warp may only touch TMEM lanes 32*(warp%4)..+31
    const int ew = warp & 3;   // TMEM lane quarter = rows 32ew..32ew+31 of [dW_f; dW_r] (or of dW_f and of dW_r)
    const int64_t ngroups = (my_tiles + kDwFlush - 1) / kDwFlush;
    if constexpr (NACC == 1) {
      float acc[C];
#pragma unroll
      for (int i = 0; i < C; ++i) acc[i] = 0.f;
      // this thread's row of the CTA's double partials: written by this thread only, L2-resident
      double2* dst = reinterpret_cast<double2*>(reinterpret_cast<double*>(p.part) + ((size_t)blockIdx.x * 128 + ew * 32 + lane) * C);
      bool first = true;
      int since = 0;
      for (int64_t grp = 0; grp < ngroups; ++grp) {
        const int a = (int)(grp & 1);
        dw_mbar_wait(&tfull[a], (uint32_t)((grp >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t taddr = tmem_base + (uint32_t)(a * TB) + ((uint32_t)(ew * 32) << 16);
#pragma unroll
        for (int c0 = 0; c0 < C; c0 += 32) {
          uint32_t v[32];
          dw_tmem_ld32(taddr + c0, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[c0 + i] += __uint_as_float(v[i]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        dw_mbar_arrive(&tempty[a]);
        if (++since == kDwRegTiles || grp + 1 == ngroups) {
#pragma unroll
          for (int q = 0; q < C / 2; ++q) {
            double2 o = make_double2((double)acc[2 * q], (double)acc[2 * q + 1]);
            if (!first) {
              const double2 prev = dst[q];
              o.x += prev.x, o.y += prev.y;
            }
            dst[q] = o;
            acc[2 * q] = 0.f, acc[2 * q + 1] = 0.f;
          }
          first = false, since = 0;
        }
      }
      if (ngroups == 0) {   // a CTA without tiles still owns a slice of the partials
#pragma unroll
        for (int q = 0; q < C / 2; ++q) dst[q] = make_double2(0.0, 0.0);
      }
    } else {
      // two 128 x C accumulators do not fit a thread's registers: the running sums live in this CTA's slice of `part`
      // (L2-resident: read-add-write by the owning thread every kDwFlush tiles)
      for (int64_t grp = 0; grp < ngroups; ++grp) {
        const int a = (int)(grp & 1);
        dw_mbar_wait(&tfull[a], (uint32_t)((grp >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int ac = 0; ac < NACC; ++ac) {
          const uint32_t taddr = tmem_base + (uint32_t)(a * TB + ac * C) + ((uint32_t)(ew * 32) << 16);
          float4* dst = reinterpret_cast<float4*>(p.part + ((size_t)blockIdx.x * dw_part_rows(C) + ac * C + ew * 32 + lane) * C);
#pragma unroll
          for (int c0 = 0; c0 < C; c0 += 32) {
            uint32_t v[32];
            dw_tmem_ld32(taddr + c0, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              float4 o = make_float4(__uint_as_float(v[q * 4]), __uint_as_float(v[q * 4 + 1]), __uint_as_float(v[q * 4 + 2]),
                                     __uint_as_float(v[q * 4 + 3]));
              if (grp > 0) f4_add(o, dst[c0 / 4 + q]);
              dst[c0 / 4 + q] = o;
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        dw_mbar_arrive(&tempty[a]);
      }
      if (ngroups == 0) {   // a CTA without tiles still owns a slice of `part`
#pragma unroll
        for (int ac = 0; ac < NACC; ++ac) {
          float4* dst = reinterpret_cast<float4*>(p.part + ((size_t)blockIdx.x * dw_part_rows(C) + ac * C + ew * 32 + lane) * C);
          for (int q = 0; q < C / 4; ++q) dst[q] = f4_zero();
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * TB) : "memory");
}

// dW_f[co][ci] = sum_cta part[cta][co][ci], dW_r = rows C..2C-1, added in CTA order in double
template <typename T>
__global__ void k_dw_tc_final(const T* __restrict__ part, int nparts, int C, int prows, float* __restrict__ dWf,
                              float* __restrict__ dWr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * C * C) return;
  const int row = i / C, col = i % C;
  double s = 0;
  for (int b = 0; b < nparts; ++b) s += (double)part[((size_t)b * prows + row) * C + col];
  if (row < C) dWf[row * C + col] = (float)s;
  else dWr[(row - C) * C + col] = (float)s;
}

static int dw_grid(int64_t M, int C) {
  const int64_t ntiles = cdiv(M, dw_tile_k(C));
  return (int)(ntiles < kNumSMs ? ntiles : kNumSMs);
}
template <int C, bool HP>
static size_t dw_smem() {
  const size_t lbo = (size_t)(dw_tile_k(C) / 4) * kDwSbo;
  const size_t stage = 2 * (dw_nacc(C) == 1 ? 4 : 2 * (C / 32)) * lbo + 2 * (C / 32) * lbo + (HP ? (C / 32) * lbo / 2 : 0);
  return (size_t)kDwStages * stage + 128 + 4 * C * sizeof(float) + 1024;
}

template <int C, bool GN, bool HP = false>
static int dw_launch(const DwParams& p, const float* Af, const float* Ar, const float* H, cudaStream_t s, int64_t ldA = 0, int64_t ldH = 0) {
  CUtensorMap tf, tr, th;
  if (int rc = make_tmap_2d_f32(&tf, Af, p.M, C, 32, dw_tile_k(C), CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, ldA)) return rc;
  if (int rc = make_tmap_2d_f32(&tr, Ar, p.M, C, 32, dw_tile_k(C), CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, ldA)) return rc;
  if (int rc = make_tmap_2d_f32(&th, H, HP ? p.M / 2 : p.M, C, 32, HP ? dw_tile_k(C) / 2 : dw_tile_k(C), CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                ldH))
    return rc;
  const size_t smem = dw_smem<C, HP>();
  TW_CUDA(cudaFuncSetAttribute(k_dw_tc<C, GN, HP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_dw_tc<C, GN, HP><<<dw_grid(p.M, C), kDwThreads, smem, s>>>(p, tf, tr, th);
  TW_LAUNCH_CHECK();
  return 0;
}

}  // namespace twowl

using namespace twowl;

extern "C" int twowl_pair_dw_supported(int32_t C) { return (C == 32 || C == 64 || C == 128) ? 1 : 0; }

template <bool GN, bool HP = false>
static int dw_dispatch(const DwParams& p, int C, const float* Af, const float* Ar, const float* H, float* dWf, float* dWr, cudaStream_t s,
                       int64_t ldA = 0, int64_t ldH = 0) {
  const int rc = C == 32   ? dw_launch<32, GN, HP>(p, Af, Ar, H, s, ldA, ldH)
                 : C == 64 ? dw_launch<64, GN, HP>(p, Af, Ar, H, s, ldA, ldH)
                           : dw_launch<128, GN, HP>(p, Af, Ar, H, s, ldA, ldH);
  if (rc) return rc;
  if (dw_nacc(C) == 1)
    k_dw_tc_final<double><<<(int)cdiv(2 * C * C, 256), 256, 0, s>>>(reinterpret_cast<const double*>(p.part), dw_grid(p.M, C), C,
                                                                   dw_part_rows(C), dWf, dWr);
  else
    k_dw_tc_final<float><<<(int)cdiv(2 * C * C, 256), 256, 0, s>>>(p.part, dw_grid(p.M, C), C, dw_part_rows(C), dWf, dWr);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_pair_dw_workspace_bytes(int64_t M, int32_t C) {
  (void)M;
  return align_up((size_t)kNumSMs * (size_t)dw_part_rows(C) * (size_t)C * (dw_nacc(C) == 1 ? sizeof(double) : sizeof(float)));
}

extern "C" int twowl_pair_dw(const float* dOf, const float* dOr, const float* rsf, const float* rsr, const float* H, int64_t M,
                             int32_t C, float* dWf, float* dWr, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(twowl_pair_dw_supported(C), "pair_dw: C=%d unsupported (32, 64 or 128)", C);
  TW_CHECK_ARG(M > 0, "pair_dw: needs M > 0");
  TW_CHECK_ARG(aligned16(dOf) && aligned16(dOr) && aligned16(H) && rsf && rsr, "pair_dw: bad pointers");
  TW_CHECK_WS(ws_bytes, twowl_pair_dw_workspace_bytes(M, C));
  DwParams p;
  memset(&p, 0, sizeof(p));
  p.rsf = rsf, p.rsr = rsr, p.M = M, p.part = (float*)ws;
  return dw_dispatch<false>(p, C, dOf, dOr, H, dWf, dWr, (cudaStream_t)stream);
}

// Column blocks of wider matrices: dOf / dOr point at a C-column block of [M, ld_dO] matrices, H at a C-column block of an
// [M, ld_H] matrix (TMA tensor maps with a row pitch) -> the corresponding [C, C] block of the weight gradients. A 256-wide layer
// is four such launches per direction pair (twowl_b200.ops.pair_dw_wide).
extern "C" int twowl_pair_dw_ld(const float* dOf, const float* dOr, const float* rsf, const float* rsr, const float* H, int64_t M,
                                int32_t C, int64_t ld_dO, int64_t ld_H, float* dWf, float* dWr, void* ws, size_t ws_bytes,
                                void* stream) {
  TW_CHECK_ARG(twowl_pair_dw_supported(C), "pair_dw_ld: C=%d unsupported (32, 64 or 128)", C);
  TW_CHECK_ARG(M > 0 && ld_dO >= C && ld_H >= C && (ld_dO & 3) == 0 && (ld_H & 3) == 0, "pair_dw_ld: pitches must be >= C and multiples of 4");
  TW_CHECK_ARG(aligned16(dOf) && aligned16(dOr) && aligned16(H) && rsf && rsr, "pair_dw_ld: bad pointers");
  TW_CHECK_WS(ws_bytes, twowl_pair_dw_workspace_bytes(M, C));
  DwParams p;
  memset(&p, 0, sizeof(p));
  p.rsf = rsf, p.rsr = rsr, p.M = M, p.part = (float*)ws;
  return dw_dispatch<false>(p, C, dOf, dOr, H, dWf, dWr, (cudaStream_t)stream, ld_dO, ld_H);
}

extern "C" int twowl_pair_dw_gn(const float* Of, const float* Or, const float* consts, const float* G, const int32_t* head,
                                const int32_t* next, float p_drop, uint64_t seed_f, uint64_t seed_r, int32_t relu, const float* rsf,
                                const float* rsr, const float* H, int32_t h_pairs, int64_t M, int32_t C, float* dOf, float* dOr,
                                float* dWf, float* dWr, void* ws, size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(twowl_pair_dw_supported(C), "pair_dw_gn: C=%d unsupported (32, 64 or 128)", C);
  TW_CHECK_ARG(M > 0 && M < 0x7fffffffLL, "pair_dw_gn: needs 0 < M < 2^31");
  TW_CHECK_ARG(h_pairs == 0 || (h_pairs == 1 && M % 2 == 0), "pair_dw_gn: h_pairs = %d needs 0, or 1 with an even M", h_pairs);
  TW_CHECK_ARG(aligned16(Of) && aligned16(Or) && aligned16(H) && aligned16(dOf) && aligned16(dOr) && aligned16(consts) && aligned16(G) &&
                   rsf && rsr && head && next,
               "pair_dw_gn: bad pointers");
  TW_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f, "pair_dw_gn: dropout p=%f outside [0,1)", p_drop);
  TW_CHECK_WS(ws_bytes, twowl_pair_dw_workspace_bytes(M, C));
  DwParams p;
  memset(&p, 0, sizeof(p));
  p.rsf = rsf, p.rsr = rsr, p.M = M, p.part = (float*)ws;
  p.consts = consts, p.G = G, p.head = head, p.next = next, p.dOf = dOf, p.dOr = dOr;
  p.thresh = p_drop > 0.f ? drop_thresh(p_drop) : 0u, p.inv_keep = 1.f / (1.f - p_drop);
  p.seed_f = seed_f, p.seed_r = seed_r, p.relu = relu;
  return h_pairs ? dw_dispatch<true, true>(p, C, Of, Or, H, dWf, dWr, (cudaStream_t)stream)
                 : dw_dispatch<true>(p, C, Of, Or, H, dWf, dWr, (cudaStream_t)stream);
}
