// Implicit-GEMM convolution for sm_100a: TMA (tiled, zero-filled halos) -> shared memory ->
// tcgen05.mma (bf16 x bf16 -> fp32 in TMEM) -> fused epilogue.  See include/diffusynth_b200.h
// (ds_conv_gemm) for the contract and the reference lines it replaces.
//
// CTA = 12 warps, persistent over output tiles:
//   warp 0      TMA producer (one elected lane): per K-block one 4-D box of the activation
//               (BK channels x Wb x Hb pixels, shifted by the tap offset; out-of-image pixels are
//               zero-filled by TMA = the conv's zero padding) and one box of the weights.
//   warp 1      MMA issuer (one elected lane): tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN,
//               K=16 per instruction, accumulator double-buffered in TMEM.
//   warp 2      TMEM allocator.
//   warps 4-11  epilogue: tcgen05.ld the accumulator (thread = pixel row), apply the folded
//               GroupNorm(1,C) scalars / bias / GELU / residual, write bf16 NHWC (or fp32 NCHW),
//               and emit (sum, sumsq) partials for the next GroupNorm.
#include "common.cuh"
#include "../../include/diffusynth_b200.h"
#include "tma.cuh"

namespace ds {

// Profiling switches (DS_CONV_DBG bitmask, tools_dev/conv_roles.py) are compiled in only with -DDS_CONV_DEBUG
// (DS_EXTRA_NVCC_FLAGS=-DDS_CONV_DEBUG python -m diffusynth_b200._build --force): the production kernels carry none of it.
#ifdef DS_CONV_DEBUG
#define DS_DBG(P) ((P).dbg)
#else
#define DS_DBG(P) 0
#endif
static constexpr int kNumThreads = 384;
static constexpr int kEpiWarp0 = 4;
static constexpr int kEpiWarps = 8;
static constexpr int kMaxStages = 8;
static constexpr int BM = 128;

struct __align__(16) ConvGemmDev {
  int N, H, W, Hb, Wb, tiles_h, tiles_w, tiles_m;
  int n_tiles_n, BN, C0, C1, cblocks0, cblocks, ntaps, groups, per_sample_w, src_batch_mod;
  int num_kb, stages, num_tiles;     // num_tiles = work items: M-tiles (cg = 1) or M-tile pairs (cg = 2)
  int cg, tiles_md, pair_flat;       // CTAs per MMA (1 or 2), tiles_m / cg, pairs over the flattened (sample, M-tile) index
  float inv_tiles_md;
  float inv_n_tiles_n, inv_tiles_m, inv_groups, inv_tiles_w, inv_Wb;   // reciprocals for fast_divmod
  unsigned long long* dbg_buf;      // DS_CONV_DBG & 64: per-CTA wait-cycle counters [grid][8]
  int dbg;                          // DS_CONV_DBG bitmask (profiling experiments): 1 = no global stores, 2 = no TMEM loads, 4 = no MMA issue
  int nacc;                         // accumulators in tensor memory: 2 (double-buffered) or 1 (two CTAs per SM, BN > 128)
  int sps;                          // K-blocks per pipeline stage (generic mode): keeps >= ~384 MMA cycles behind every barrier round trip
  unsigned stage_a_bytes, stage_b_bytes;
  int Cout, Cout_pad;
  const float2* stats_in; int stats_in_slots; float out_inv_count, eps;
  const float* e1; const float* e2; int ncls;
  const float* sbias; int sbias_stride; int act;
  const act_t* residual; long long res_sn, res_sh, res_sw;
  act_t* out; long long out_sn, out_sh, out_sw; long long out_goff[DS_MAX_GROUPS];
  float* out_f32;
  float2* stats_out; int stats_slots;
  ds_conv_tap taps[DS_MAX_GROUPS][DS_MAX_TAPS];
};

struct TmaMaps {
  CUtensorMap a[2][4];   // [source][view]
  CUtensorMap b;
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// One lane of a converged warp (the lowest): the producer and MMA warps run their loops warp-uniformly and predicate only the
// TMA / MMA / arrive instructions with this, so the loop state stays in uniform registers (a loop under `if (lane == 0)` makes
// the compiler re-broadcast every operand of every tensor instruction).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
// mbar_wait that also accumulates the cycles spent waiting (profiling builds of the role loops: DS_CONV_DBG & 64)
__device__ __forceinline__ void mbar_wait_timed(uint64_t* bar, uint32_t parity, bool timed, long long& acc) {
  if (!timed) { mbar_wait_warp(bar, parity); return; }
  const long long t0 = clock64();
  mbar_wait_warp(bar, parity);
  acc += clock64() - t0;
}
// ---- 2-CTA (cta_group::2) variants: one MMA instruction drives the tensor cores of both SMs of a cluster pair (M = 256: each CTA
// holds its own 128 activation rows and HALF of the weight tile), issued by the even ("leader") CTA only.
static constexpr uint32_t kPeerMask = 0xFEFFFFFFu;     // clears the CTA-rank bit of a shared::cluster address -> the leader's copy
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs once all previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
// TMA loads of either CTA of the pair that report their bytes to the LEADER's barrier
__device__ __forceinline__ void tma_load_4d_2cta(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar) & kPeerMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2cta(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar) & kPeerMask), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Plain arrive on the leader CTA's copy of the barrier.  RELAXED: the barrier only hands the tensor-memory accumulator back to the MMA
// warp, and the epilogue's reads of it are complete (tcgen05.wait::ld) and ordered (tcgen05.fence::before_thread_sync) before the
// arrive.  A .release.cluster arrive makes ptxas emit a cluster-scope memory barrier first, which waits for the tile's output stores
// to be acknowledged by L2: ncu showed 25 % of the GELU epilogue's stall samples on that MEMBAR / ERRBAR pair.
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerMask) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; both operands K-major, described by 64-bit shared-memory descriptors.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): rows of BK bf16 = one swizzle span
// (64 B or 128 B), 8-row groups SBO bytes apart; version 1 (Blackwell); layout type 2 = SWIZZLE_128B, 4 = SWIZZLE_64B.
template <int BK>
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr) {
  constexpr uint64_t row_bytes = BK * 2;
  constexpr uint64_t sbo = (8 * row_bytes) >> 4;
  constexpr uint64_t layout = (BK == 64) ? 2ull : 4ull;
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}

// ---------------------------------------------------------------------------------------------
// Kernel
// ---------------------------------------------------------------------------------------------
struct TileCoord { int n, g, th, tw, nt, slot; };

// x / d and x % d for 0 <= x < 2^22, 1 <= d: float reciprocal estimate + one correction step (6 instructions instead of the
// ~25 of an integer division; the tile decode runs once per tile in every role warp).
__device__ __forceinline__ void fast_divmod(int x, int d, float inv_d, int& q, int& r) {
  q = __float2int_rz(((float)x + 0.5f) * inv_d);
  r = x - q * d;
  if (r < 0) { --q; r += d; }
  else if (r >= d) { ++q; r -= d; }
}

// tile = work index of the CTA (CG = 1) or of the CTA pair (CG = 2: the pair owns M-tiles 2m', 2m'+1 of one (sample, group, n-tile))
__device__ __forceinline__ TileCoord decode_tile(const ConvGemmDev& P, int tile, int rank) {
  TileCoord t;
  int r, m;
  fast_divmod(tile, P.n_tiles_n, P.inv_n_tiles_n, r, t.nt);
  if (P.cg == 2 && P.pair_flat) {
    // pairs run over the flattened (sample, M-tile) index: also covers an odd number of M-tiles per sample (groups == 1)
    fast_divmod(2 * r + rank, P.tiles_m, P.inv_tiles_m, t.n, m);
    t.g = 0;
  } else {
    int r2;
    fast_divmod(r, P.tiles_md, P.inv_tiles_md, r2, m);
    m = m * P.cg + rank;
    fast_divmod(r2, P.groups, P.inv_groups, t.n, t.g);
  }
  fast_divmod(m, P.tiles_w, P.inv_tiles_w, t.th, t.tw);
  t.slot = (t.g * P.tiles_m + m) * P.n_tiles_n + t.nt;
  return t;
}

// tcgen05.wait::ld with the destination registers as in/out operands, so that no use of them can be scheduled
// above the wait.
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {          // read-only tables: may be scheduled freely
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ int4 lds_i4(uint32_t addr) {
  int4 v;
  asm("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 lds_f4_volatile(uint32_t addr) { // per-tile buffers rewritten by the same warp
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// GELU(x) = relu(x) - 0.5 |x| q(|x|),  q = poly(t) t exp(-x^2/2),  t = 1/(1 + p |x|/sqrt2)   (Abramowitz-Stegun 7.1.26,
// |erf error| <= 1.5e-7; the 0.5 is folded into the coefficients): 2 MUFU + 13 FP32 ops per value.
// GELU on 16 values, written stage by stage over groups of 8 so that the 8 independent dependency chains interleave
// (ptxas serialises a per-element formulation when registers are tight: ~80 cycles per element at 2 warps per scheduler).
__device__ __forceinline__ void gelu16(float (&v)[16]) {
#pragma unroll
  for (int g = 0; g < 16; g += 8) {
    float ax[8], t[8], e[8], p[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) ax[j] = fabsf(v[g + j]);
#pragma unroll
    for (int j = 0; j < 8; ++j) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t[j]) : "f"(fmaf(0.3275911f * 0.70710678118654752f, ax[j], 1.0f)));
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float w = ax[j] * 0.84932180028801904f; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[j]) : "f"(-w * w)); }
#pragma unroll
    for (int j = 0; j < 8; ++j) p[j] = fmaf(0.5f * 1.061405429f, t[j], 0.5f * -1.453152027f);
#pragma unroll
    for (int j = 0; j < 8; ++j) p[j] = fmaf(p[j], t[j], 0.5f * 1.421413741f);
#pragma unroll
    for (int j = 0; j < 8; ++j) p[j] = fmaf(p[j], t[j], 0.5f * -0.284496736f);
#pragma unroll
    for (int j = 0; j < 8; ++j) p[j] = fmaf(p[j], t[j], 0.5f * 0.254829592f);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[g + j] = fmaxf(v[g + j], 0.0f) - ax[j] * (p[j] * t[j] * e[j]);
  }
}

// Packed fp32x2 arithmetic (sm_100 FFMA2 / FMUL2 / FADD2: two IEEE fp32 operations per issue slot).  The GELU epilogue is bound by
// the issue slots of its two warps per scheduler (376 instructions per 16-column chunk, 68 % of the slots busy: measured
// 1.1 k cycles per chunk), so the fold, the GELU polynomial and the statistics run on register pairs.
typedef unsigned long long f2_t;
__device__ __forceinline__ f2_t f2_pack(float lo, float hi) { f2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void f2_unpack(f2_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2_t f2_fma(f2_t a, f2_t b, f2_t c) { f2_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f2_t f2_mul(f2_t a, f2_t b) { f2_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2_t f2_add(f2_t a, f2_t b) { f2_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// gelu16 on 8 register pairs (same formula, same constants): per pair 2 abs/neg + 2 max + 4 MUFU stay scalar, the 10 multiply-adds are
// packed.  Stage by stage over 4 pairs so that 8 independent chains interleave.
__device__ __forceinline__ void gelu16_f2(f2_t (&v)[8]) {
  const f2_t kP = f2_pack(-0.3275911f * 0.70710678118654752f, -0.3275911f * 0.70710678118654752f);      // times -|x|
  const f2_t kOne = f2_pack(1.0f, 1.0f);
  const f2_t kW = f2_pack(0.84932180028801904f, 0.84932180028801904f);
  const f2_t a5 = f2_pack(0.5f * 1.061405429f, 0.5f * 1.061405429f), a4 = f2_pack(0.5f * -1.453152027f, 0.5f * -1.453152027f);
  const f2_t a3 = f2_pack(0.5f * 1.421413741f, 0.5f * 1.421413741f), a2 = f2_pack(0.5f * -0.284496736f, 0.5f * -0.284496736f);
  const f2_t a1 = f2_pack(0.5f * 0.254829592f, 0.5f * 0.254829592f);
#pragma unroll
  for (int g = 0; g < 8; g += 4) {
    f2_t nax[4], relu[4], t[4], e[4], p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x0, x1;
      f2_unpack(v[g + j], x0, x1);
      nax[j] = f2_pack(-fabsf(x0), -fabsf(x1));
      relu[j] = f2_pack(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f));
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float d0, d1, t0, t1;
      f2_unpack(f2_fma(kP, nax[j], kOne), d0, d1);
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
      t[j] = f2_pack(t0, t1);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const f2_t w = f2_mul(nax[j], kW);
      float q0, q1, e0, e1;
      f2_unpack(f2_mul(w, w), q0, q1);
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-q0));
      asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-q1));
      e[j] = f2_pack(e0, e1);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = f2_fma(a5, t[j], a4);
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = f2_fma(p[j], t[j], a3);
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = f2_fma(p[j], t[j], a2);
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = f2_fma(p[j], t[j], a1);
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = f2_mul(f2_mul(p[j], t[j]), e[j]);
#pragma unroll
    for (int j = 0; j < 4; ++j) v[g + j] = f2_fma(nax[j], p[j], relu[j]);      // relu(x) - |x| * (0.5 poly(t) t e)
  }
}

#ifdef DS_OPERANDS_BF16
__device__ __forceinline__ uint32_t pack16_epi(float lo, float hi) { return pack16(lo, hi); }
#else
__device__ __forceinline__ uint32_t pack16_epi(float lo, float hi) {   // one F2FP.SATFINITE instead of clamp + convert
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
#endif

// One pipeline stage = sps x (A tap tile | B tile).  Warp roles: 0 = activation (A) TMA producer, 1 = MMA issuer, 2 = TMEM
// allocator, then weight (B) TMA producer, 3 = statistics publisher, 4-11 = epilogue.  The two producers split the per-K-block
// scalar work (barrier probe + coordinates + TMA issue), which otherwise bounds the kernel on one thread; the A producer
// reads its per-K-block coordinates (tensor map, channel offset, tap shift) from a table built once in shared memory.
// EPI specialises the epilogue so that every instantiation carries only the code it runs (the generic kernel is ~9000 SASS
// instructions and the role warps evict each other from the instruction cache): 0 = everything (fp32 / ragged outputs),
// 1 = 16-bit output with full chunks, no activation, no residual (the 1x1 convolutions), 2 = + GELU (conv1), 3 = + residual (conv2),
// 4 = as 1 without GroupNorm fold and per-sample bias (to_out, res_conv: value = acc + e2[col]; a third of the instructions of 1).
// EPI = 4 with one CTA per MMA (the plain 1x1 convolutions to_out / res_conv: short K loops, latency-bound epilogues) is compiled for
// TWO resident CTAs per SM (<= 80 registers; the launcher then gives each CTA half of the shared memory and at most 256 TMEM columns):
// while one CTA waits for its accumulator or its stores, the other one runs.
template <int BK, int CG, int EPI>
__global__ void __launch_bounds__(kNumThreads, (EPI == 4 && CG == 1) ? 2 : 1)
conv_gemm_kernel(const __grid_constant__ TmaMaps maps, const __grid_constant__ ConvGemmDev P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages x sps x (A | B)] | barriers | stats partials | sbias | tables e2, e1 | K-block table
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const unsigned sub_bytes = P.stage_a_bytes + P.stage_b_bytes;
  const unsigned stage_bytes = (unsigned)P.sps * sub_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full = empty_bar + kMaxStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* stats_full = tmem_empty + 2;
  uint64_t* stats_empty = stats_full + 2;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(stats_empty + 2);
  float2* s_stats = reinterpret_cast<float2*>(tmem_base_smem + 4);          // [2][kEpiWarps]
  float* s_sb = reinterpret_cast<float*>(s_stats + 2 * kEpiWarps);           // [kEpiWarps][128] per-sample bias of the current tile
  float* s_e2 = s_sb + kEpiWarps * 128;
  float* s_e1 = s_e2 + P.ncls * P.Cout_pad;
  int4* s_kbt = reinterpret_cast<int4*>(s_e1 + P.ncls * P.Cout_pad);         // [groups][num_kb]: {tensor-map byte offset, channel, dx, dy}

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = (CG == 2) ? (int)cluster_ctarank() : 0;           // 0 = leader of the pair
  const int w_first = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int w_step = (CG == 2) ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int acc_cols = P.nacc * P.BN;      // nacc accumulators of BN columns (2 = double-buffered; 1 = two CTAs per SM share the tensor memory)
  const uint32_t tmem_cols = (acc_cols <= 32) ? 32u : (acc_cols <= 64) ? 64u : (acc_cols <= 128) ? 128u : (acc_cols <= 256) ? 256u : 512u;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < 2; ++s)
      for (int v = 0; v < 4; ++v) prefetch_tmap(&maps.a[s][v]);
    prefetch_tmap(&maps.b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full_bar[s], 2);          // one arrive.expect_tx from each producer
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], CG * kEpiWarps);      // CG = 2: the leader's copy collects the epilogue warps of both CTAs
      mbar_init(&stats_full[a], kEpiWarps);
      mbar_init(&stats_empty[a], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) { if (CG == 2) tmem_alloc_2cta(tmem_base_smem, tmem_cols); else tmem_alloc(tmem_base_smem, tmem_cols); }
  for (int i = threadIdx.x; i < P.ncls * P.Cout_pad; i += kNumThreads) {
    s_e2[i] = __ldg(P.e2 + i);
    s_e1[i] = P.e1 ? __ldg(P.e1 + i) : 0.f;
  }
  for (int i = threadIdx.x; i < P.groups * P.num_kb; i += kNumThreads) {
    const int g = i / P.num_kb, kb = i - g * P.num_kb;
    const int tap = kb / P.cblocks, cb = kb - tap * P.cblocks;
    const ds_conv_tap tp = P.taps[g][tap];
    const int src = cb < P.cblocks0 ? 0 : 1;
    s_kbt[i] = make_int4((src * 4 + tp.view) * (int)sizeof(CUtensorMap), (src == 0 ? cb : cb - P.cblocks0) * BK, tp.dx, tp.dy);
  }
  // (everything above reads only launch parameters and weight tables: it overlaps the tail of the previous kernel)
  pdl_launch_dependents();
  pdl_wait();
  tcgen05_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();        // the peer's barriers are initialised before anything is signalled across the pair
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;
  const bool timed = (DS_DBG(P) & 64) != 0;

  if (warp == 0) {
    // ================================ activation (A) producer: warp-uniform, one elected lane issues =======================
    long long w_empty = 0;
    const long long t_begin = clock64();
    const uint8_t* map_base = reinterpret_cast<const uint8_t*>(&maps.a[0][0]);
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = w_first; tile < P.num_tiles; tile += w_step) {
      const TileCoord t = decode_tile(P, tile, rank);
      const int nsrc = P.src_batch_mod > 0 ? (t.n % P.src_batch_mod) : t.n;
      const int h0 = t.th * P.Hb, w0 = t.tw * P.Wb;
      const uint32_t kbt = smem_u32(s_kbt + t.g * P.num_kb);      // shared-space address: the entries are read with LDS
      for (int kb = 0; kb < P.num_kb; kb += P.sps) {
        const int nsub = (P.num_kb - kb) < P.sps ? (P.num_kb - kb) : P.sps;
        int4 e[4];                                                   // this stage's entries, fetched before the barrier probe
#pragma unroll
        for (int j = 0; j < 4; ++j) e[j] = lds_i4(kbt + (uint32_t)(kb + (j < nsub ? j : 0)) * 16u);
        mbar_wait_timed(&empty_bar[stage], phase ^ 1u, timed, w_empty);
        if (elect_one_sync()) {
          uint8_t* sa = smem + (size_t)stage * stage_bytes;
          if (rank == 0) mbar_expect_tx(&full_bar[stage], (unsigned)(CG * nsub) * P.stage_a_bytes);      // the pair's activation bytes
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < nsub) {
              const CUtensorMap* mp = reinterpret_cast<const CUtensorMap*>(map_base + e[j].x);
              const int ns = e[j].x < 4 * (int)sizeof(CUtensorMap) ? nsrc : t.n;      // the batch modulus applies to source 0 only
              if (CG == 2) tma_load_4d_2cta(sa, mp, &full_bar[stage], e[j].y, w0 + e[j].z, h0 + e[j].w, ns);
              else tma_load_4d(sa, mp, &full_bar[stage], e[j].y, w0 + e[j].z, h0 + e[j].w, ns);
              sa += sub_bytes;
            }
          }
        }
        __syncwarp();
        if (++stage == P.stages) { stage = 0; phase ^= 1u; }
      }
    }
    if (timed && lane == 0) { P.dbg_buf[blockIdx.x * 16 + 0] = (unsigned long long)w_empty; P.dbg_buf[blockIdx.x * 16 + 1] = (unsigned long long)(clock64() - t_begin); }
  } else if (warp == 2) {
    // ================================ weight (B) producer ================================
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = w_first; tile < P.num_tiles; tile += w_step) {
      const TileCoord t = decode_tile(P, tile, rank);
      const int wz = P.per_sample_w ? t.n : t.g;
      const int n0 = t.nt * P.BN + rank * (P.BN / CG);       // CG = 2: each CTA stages its half of the weight rows
      for (int kb = 0; kb < P.num_kb; kb += P.sps) {
        const int nsub = (P.num_kb - kb) < P.sps ? (P.num_kb - kb) : P.sps;
        mbar_wait_warp(&empty_bar[stage], phase ^ 1u);
        if (elect_one_sync()) {
          uint8_t* sb = smem + (size_t)stage * stage_bytes + P.stage_a_bytes;
          if (rank == 0) mbar_expect_tx(&full_bar[stage], (unsigned)(CG * nsub) * P.stage_b_bytes);
          for (int j = 0; j < nsub; ++j) {
            if (CG == 2) tma_load_3d_2cta(sb, &maps.b, &full_bar[stage], (kb + j) * BK, n0, wz);
            else tma_load_3d(sb, &maps.b, &full_bar[stage], (kb + j) * BK, n0, wz);
            sb += sub_bytes;
          }
        }
        __syncwarp();
        if (++stage == P.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ================================ MMA issuer (warp-uniform; one elected lane issues; leader CTA only) ====================
    // instruction descriptor: D=f32 (bit 4), A/B format (bits 7-9, 10-12), K-major both, N>>3 at 17, M>>4 at 24
    const uint32_t fmt = kOperandIsFp16 ? 0u : 1u;   // F16F32Format: 0 = f16, 1 = bf16
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(P.BN >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    long long w_full = 0, w_tmem = 0, c_fence = 0, c_issue = 0, c_commit = 0;
    const long long t_begin = clock64();
    for (int tile = w_first; tile < P.num_tiles; tile += w_step) {
      mbar_wait_timed(&tmem_empty[acc], acc_phase ^ 1u, timed, w_tmem);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * P.BN);
      uint32_t accum = 0;
      for (int kb = 0; kb < P.num_kb; kb += P.sps) {
        const int nsub = (P.num_kb - kb) < P.sps ? (P.num_kb - kb) : P.sps;
        mbar_wait_timed(&full_bar[stage], phase, timed, w_full);
        long long tq0 = 0, tq1 = 0, tq2 = 0;
        if (timed) tq0 = clock64();
        tcgen05_fence_after();
        if (timed) { tq1 = clock64(); c_fence += tq1 - tq0; }
        if (elect_one_sync()) {
          uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
          for (int j = 0; j < nsub; ++j) {
            const uint64_t adesc = make_kmajor_desc<BK>(sa);
            const uint64_t bdesc = make_kmajor_desc<BK>(sa + P.stage_a_bytes);
            if (!(DS_DBG(P) & 4)) {
              // advance 16 elements (32 bytes) along K inside the swizzle span: +2 in the 16-byte address field
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                if (CG == 2) umma_f16_2cta(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (k > 0 || j > 0) ? 1u : accum);
                else umma_f16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (k > 0 || j > 0) ? 1u : accum);
              }
            }
            sa += sub_bytes;
          }
          if (timed) { tq2 = clock64(); c_issue += tq2 - tq1; }
          if (CG == 2) umma_commit_2cta(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);   // frees the smem slot (of both CTAs) when these MMAs retire
          if (timed) c_commit += clock64() - tq2;
        }
        __syncwarp();
        accum = 1u;
        if (++stage == P.stages) { stage = 0; phase ^= 1u; }
      }
      if (elect_one_sync()) { if (CG == 2) umma_commit_2cta(&tmem_full[acc]); else umma_commit(&tmem_full[acc]); }       // accumulator complete
      __syncwarp();
      if (++acc == P.nacc) { acc = 0; acc_phase ^= 1u; }
    }
    if (timed && lane == 0) {
      P.dbg_buf[blockIdx.x * 16 + 2] = (unsigned long long)w_full; P.dbg_buf[blockIdx.x * 16 + 3] = (unsigned long long)w_tmem;
      P.dbg_buf[blockIdx.x * 16 + 4] = (unsigned long long)(clock64() - t_begin);
      P.dbg_buf[blockIdx.x * 16 + 8] = (unsigned long long)c_fence; P.dbg_buf[blockIdx.x * 16 + 9] = (unsigned long long)c_issue;
      P.dbg_buf[blockIdx.x * 16 + 10] = (unsigned long long)c_commit;
    }
  } else if (warp == 3) {
    // ================================ statistics publisher =========================
    // Sums the 8 epilogue-warp partials of each tile (fixed order), writes one slot per tile and runs the
    // last-arriver reduction, so the epilogue warps never wait on a memory fence or an atomic.
    if (P.stats_out != nullptr) {
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = w_first; tile < P.num_tiles; tile += w_step) {
        const TileCoord t = decode_tile(P, tile, rank);
        mbar_wait_warp(&stats_full[acc], acc_phase);
        float s = 0.f, q = 0.f;
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < kEpiWarps; ++i) { const float2 v = s_stats[acc * kEpiWarps + i]; s += v.x; q += v.y; }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&stats_empty[acc]);
        stats_publish(stats_sample(P.stats_out, P.stats_slots, t.n), P.stats_slots, t.slot, s, q, P.out_inv_count, P.eps, lane);
        if (++acc == P.nacc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ================================ epilogue ====================================
    const int ew = warp - kEpiWarp0;       // 0..7
    const int lane_grp = warp & 3;         // TMEM lanes [32*lane_grp, +32) are the ones this warp may read
    const int col_half = ew >> 2;          // two warps share a lane group and split the columns
    const int row = lane_grp * 32 + lane;  // accumulator row = pixel inside the tile
    const int chunks = P.BN / 16;          // 16-column chunks
    const int chunk_lo = col_half == 0 ? 0 : (chunks + 1) / 2;
    const int chunk_hi = col_half == 0 ? (chunks + 1) / 2 : chunks;
    int ph, pw;
    fast_divmod(row, P.Wb, P.inv_Wb, ph, pw);
    int acc = 0;
    uint32_t acc_phase = 0;
    // per-sample bias (to_qkv's label_query/label_key): this warp's column range, fetched one tile ahead into
    // registers and parked in shared memory while the tile is processed
    float* my_sb = s_sb + ew * 128;
    const int sb_cols = (chunk_hi - chunk_lo) * 16;
    float sb_next[4] = {0.f, 0.f, 0.f, 0.f};
    float2 mr_next = make_float2(0.f, 1.f);      // (mean, rstd) of the next tile's sample, fetched one tile ahead like the bias
    auto fetch_sbias = [&](int tile_idx) {
      if (tile_idx >= P.num_tiles || (P.sbias == nullptr && P.stats_in == nullptr)) return;
      const TileCoord tt = decode_tile(P, tile_idx, rank);
      if (P.stats_in != nullptr) {
        const int nsrc = P.src_batch_mod > 0 ? (tt.n % P.src_batch_mod) : tt.n;
        mr_next = __ldg(stats_sample(P.stats_in, P.stats_in_slots, nsrc));
      }
      if (P.sbias == nullptr) return;
      const float* src = P.sbias + (size_t)tt.n * P.sbias_stride + tt.nt * P.BN + chunk_lo * 16;
#pragma unroll
      for (int i = 0; i < 4; ++i) sb_next[i] = (lane + 32 * i < sb_cols) ? __ldg(src + lane + 32 * i) : 0.f;
    };
    if (EPI != 4) fetch_sbias(w_first);
    const bool epi_timed = (DS_DBG(P) & 64) != 0;
    long long epi_wait = 0;
    const long long epi_begin = clock64();
    long long e_pro = 0, e_chunks = 0, e_tail = 0;
    for (int tile = w_first; tile < P.num_tiles; tile += w_step) {
      long long te0 = 0, te1 = 0, te2 = 0;
      if (epi_timed) te0 = clock64();
      const TileCoord t = decode_tile(P, tile, rank);
      const int h = t.th * P.Hb + ph, w = t.tw * P.Wb + pw;
      const float mean = mr_next.x, rstd = mr_next.y;
      const float nmr = -mean * rstd;
      const bool valid = (h < P.H) && (w < P.W);
      const int col0 = t.nt * P.BN + chunk_lo * 16;        // first global output channel of this warp's column range
      if (EPI != 4 && P.sbias != nullptr) {
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) my_sb[lane + 32 * i] = sb_next[i];
        __syncwarp();
      }
      if (EPI != 4) fetch_sbias(tile + w_step);
      int cls = 0;
      if (P.ncls == 9) cls = (h == 0 ? 0 : (h == P.H - 1 ? 2 : 1)) * 3 + (w == 0 ? 0 : (w == P.W - 1 ? 2 : 1));
      const bool use_e1 = EPI != 4 && P.e1 != nullptr, use_sb = EPI != 4 && P.sbias != nullptr, do_stats = P.stats_out != nullptr;
      // running addresses, advanced by one 16-column chunk at a time: 32-bit shared-space addresses for the tables (so the
      // loads are LDS with immediate offsets, not generic LD), element pointers for the tensors
      uint32_t e2_s = smem_u32(s_e2) + (uint32_t)(cls * P.Cout_pad + col0) * 4u;
      uint32_t e1_s = smem_u32(s_e1) + (uint32_t)(cls * P.Cout_pad + col0) * 4u;
      uint32_t sb_s = smem_u32(my_sb);
      act_t* out_p = P.out ? P.out + (P.out_goff[t.g] + (long long)t.n * P.out_sn + (long long)h * P.out_sh + (long long)w * P.out_sw + col0) : nullptr;
      const act_t* res_p = P.residual ? P.residual + ((long long)t.n * P.res_sn + (long long)h * P.res_sh + (long long)w * P.res_sw + col0) : nullptr;
      float* o32_p = P.out_f32 ? P.out_f32 + (((size_t)t.n * P.Cout + col0) * P.H + h) * P.W + w : nullptr;
      const size_t o32_stride = (size_t)P.H * P.W;
      const bool has_res = res_p != nullptr && valid;
      int cols_left = P.Cout - col0;                       // real (unpadded) output channels from col0 on
      float psum = 0.f, psq = 0.f;
      f2_t psum2 = 0ull, psq2 = 0ull;      // EPI = 2: packed partial sums (even / odd columns), merged after the chunks

      // one 16-column chunk: folded-GroupNorm scalars, bias, activation, residual, statistics, store.
      // r = accumulator values, ra/rb = prefetched residual.  Advances the running addresses.
      auto finish_chunk = [&](const uint32_t* r, const uint4& ra, const uint4& rb) {
        float v[16];
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const float4 b4 = lds_f4(e2_s + 16u * q4);
          v[4 * q4 + 0] = fmaf(__uint_as_float(r[4 * q4 + 0]), rstd, b4.x);
          v[4 * q4 + 1] = fmaf(__uint_as_float(r[4 * q4 + 1]), rstd, b4.y);
          v[4 * q4 + 2] = fmaf(__uint_as_float(r[4 * q4 + 2]), rstd, b4.z);
          v[4 * q4 + 3] = fmaf(__uint_as_float(r[4 * q4 + 3]), rstd, b4.w);
        }
        if (use_e1) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const float4 a4 = lds_f4(e1_s + 16u * q4);
            v[4 * q4 + 0] = fmaf(nmr, a4.x, v[4 * q4 + 0]);
            v[4 * q4 + 1] = fmaf(nmr, a4.y, v[4 * q4 + 1]);
            v[4 * q4 + 2] = fmaf(nmr, a4.z, v[4 * q4 + 2]);
            v[4 * q4 + 3] = fmaf(nmr, a4.w, v[4 * q4 + 3]);
          }
        }
        if (use_sb) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const float4 a4 = lds_f4_volatile(sb_s + 16u * q4);
            v[4 * q4 + 0] += a4.x; v[4 * q4 + 1] += a4.y; v[4 * q4 + 2] += a4.z; v[4 * q4 + 3] += a4.w;
          }
        }
        if (P.act == 1) gelu16(v);
        if (valid && cols_left > 0) {
          if (has_res) {
            const uint32_t rr[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              v[2 * j] += lo16(rr[j]);
              v[2 * j + 1] += hi16(rr[j]);
            }
          }
          if (do_stats) {
            if (cols_left >= 16) {
#pragma unroll
              for (int j = 0; j < 16; ++j) { psum += v[j]; psq = fmaf(v[j], v[j], psq); }
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (j < cols_left) { psum += v[j]; psq = fmaf(v[j], v[j], psq); }
            }
          }
          if (out_p != nullptr && !(DS_DBG(P) & 1)) {           // Cout % 16 == 0 is enforced for 16-bit outputs
            uint4 a, b;
            a.x = pack16_epi(v[0], v[1]);   a.y = pack16_epi(v[2], v[3]);
            a.z = pack16_epi(v[4], v[5]);   a.w = pack16_epi(v[6], v[7]);
            b.x = pack16_epi(v[8], v[9]);   b.y = pack16_epi(v[10], v[11]);
            b.z = pack16_epi(v[12], v[13]); b.w = pack16_epi(v[14], v[15]);
            stg_256(out_p, a, b);
          }
          if (o32_p != nullptr) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < cols_left) o32_p[(size_t)j * o32_stride] = v[j];
          }
        }
        e2_s += 64u; e1_s += 64u; sb_s += 64u;
        if (out_p) out_p += 16;
        if (o32_p) o32_p += 16 * o32_stride;
        cols_left -= 16;
      };
      const uint32_t t_row = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(acc * P.BN + chunk_lo * 16);
      auto issue_chunk = [&](int c, uint32_t (&r)[16]) {      // c = chunk index inside this warp's column range
        if (DS_DBG(P) & 2) {
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = 0x3f800000u + j;
          return;
        }
        tmem_ld_32x32b_x16(t_row + (uint32_t)(c * 16), r);
      };
      // software pipeline at chunk granularity: while chunk c is being finished, the TMEM load and the residual fetch of
      // chunk c+1 are in flight (the first residual fetch is issued before waiting for the accumulator)
      uint32_t ra_[16], rb_[16];
      uint4 qa[2], qb[2];
      const int nch = chunk_hi - chunk_lo;
      const int cols0 = cols_left;
      auto fetch_res = [&](int c, uint4 (&rr)[2]) {
        rr[0] = rr[1] = make_uint4(0, 0, 0, 0);
        if ((EPI == 0 || EPI == 3) && has_res && cols0 - 16 * c > 0) {
          ldg_256(res_p + 16 * c, rr[0], rr[1]);
        }
      };
      if (nch > 0) fetch_res(0, qa);
      if (epi_timed) { te1 = clock64(); e_pro += te1 - te0; }
      mbar_wait_timed(&tmem_full[acc], acc_phase, epi_timed, epi_wait);
      if (epi_timed) te1 = clock64();
      tcgen05_fence_after();
      if (nch > 0) issue_chunk(0, ra_);
      // Main path (16-bit output, full chunks): all table reads of a chunk are issued together, so they overlap instead of
      // queueing behind each other through reused registers (what bounded the store-bound 1x1 convolutions).
      const bool lean = EPI != 0 || (out_p != nullptr && o32_p == nullptr && cols_left >= 16 * nch && !(DS_DBG(P) & 1));
      if (lean) {
        auto lean_chunk = [&](const uint32_t* r, const uint4& ra, const uint4& rb) {
          float4 t2[4], t1[4], tb[4];
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) t2[q4] = lds_f4(e2_s + 16u * q4);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) t1[q4] = (EPI == 2 || use_e1) ? lds_f4(e1_s + 16u * q4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) tb[q4] = (EPI != 2 && use_sb) ? lds_f4_volatile(sb_s + 16u * q4) : make_float4(0.f, 0.f, 0.f, 0.f);
          if (EPI == 2) {
            // GELU epilogue on register pairs: fold, GELU, statistics and the 16-bit pack (see gelu16_f2)
            const f2_t rstd2 = f2_pack(rstd, rstd), nmr2 = f2_pack(nmr, nmr);
            f2_t v2[8];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              // (the launcher selects EPI = 2 only for convolutions with a GroupNorm fold and without per-sample bias)
              const f2_t c0 = f2_fma(nmr2, f2_pack(t1[q4].x, t1[q4].y), f2_pack(t2[q4].x, t2[q4].y));
              const f2_t c1 = f2_fma(nmr2, f2_pack(t1[q4].z, t1[q4].w), f2_pack(t2[q4].z, t2[q4].w));
              v2[2 * q4 + 0] = f2_fma(f2_pack(__uint_as_float(r[4 * q4 + 0]), __uint_as_float(r[4 * q4 + 1])), rstd2, c0);
              v2[2 * q4 + 1] = f2_fma(f2_pack(__uint_as_float(r[4 * q4 + 2]), __uint_as_float(r[4 * q4 + 3])), rstd2, c1);
            }
            gelu16_f2(v2);
            if (valid) {
              uint32_t pk[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                if (do_stats) { psum2 = f2_add(psum2, v2[j]); psq2 = f2_fma(v2[j], v2[j], psq2); }
                float lo, hi;
                f2_unpack(v2[j], lo, hi);
                pk[j] = pack16_epi(lo, hi);
              }
              stg_256(out_p, make_uint4(pk[0], pk[1], pk[2], pk[3]), make_uint4(pk[4], pk[5], pk[6], pk[7]));
            }
            e2_s += 64u; e1_s += 64u; sb_s += 64u; out_p += 16;
            return;
          }
          float v[16];
          if (EPI == 4) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              v[4 * q4 + 0] = __uint_as_float(r[4 * q4 + 0]) + t2[q4].x; v[4 * q4 + 1] = __uint_as_float(r[4 * q4 + 1]) + t2[q4].y;
              v[4 * q4 + 2] = __uint_as_float(r[4 * q4 + 2]) + t2[q4].z; v[4 * q4 + 3] = __uint_as_float(r[4 * q4 + 3]) + t2[q4].w;
            }
          } else
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            v[4 * q4 + 0] = fmaf(__uint_as_float(r[4 * q4 + 0]), rstd, fmaf(nmr, t1[q4].x, t2[q4].x) + tb[q4].x);
            v[4 * q4 + 1] = fmaf(__uint_as_float(r[4 * q4 + 1]), rstd, fmaf(nmr, t1[q4].y, t2[q4].y) + tb[q4].y);
            v[4 * q4 + 2] = fmaf(__uint_as_float(r[4 * q4 + 2]), rstd, fmaf(nmr, t1[q4].z, t2[q4].z) + tb[q4].z);
            v[4 * q4 + 3] = fmaf(__uint_as_float(r[4 * q4 + 3]), rstd, fmaf(nmr, t1[q4].w, t2[q4].w) + tb[q4].w);
          }
          if (EPI == 0 ? P.act == 1 : EPI == 2) gelu16(v);
          if (valid) {
            if ((EPI == 0 || EPI == 3) && has_res) {
              const uint32_t rr[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[2 * j] += lo16(rr[j]); v[2 * j + 1] += hi16(rr[j]); }
            }
            if (do_stats) {
#pragma unroll
              for (int j = 0; j < 16; ++j) { psum += v[j]; psq = fmaf(v[j], v[j], psq); }
            }
            uint4 a, b;
            a.x = pack16_epi(v[0], v[1]);   a.y = pack16_epi(v[2], v[3]);
            a.z = pack16_epi(v[4], v[5]);   a.w = pack16_epi(v[6], v[7]);
            b.x = pack16_epi(v[8], v[9]);   b.y = pack16_epi(v[10], v[11]);
            b.z = pack16_epi(v[12], v[13]); b.w = pack16_epi(v[14], v[15]);
            stg_256(out_p, a, b);
          }
          e2_s += 64u; e1_s += 64u; sb_s += 64u; out_p += 16;
        };
        for (int c = 0; c < nch; c += 2) {
          tmem_ld_wait16(ra_);
          if (c + 1 < nch) { issue_chunk(c + 1, rb_); fetch_res(c + 1, qb); }
          lean_chunk(ra_, qa[0], qa[1]);
          if (c + 1 < nch) {
            tmem_ld_wait16(rb_);
            if (c + 2 < nch) { issue_chunk(c + 2, ra_); fetch_res(c + 2, qa); }
            lean_chunk(rb_, qb[0], qb[1]);
          }
        }
      } else if (EPI == 0) {
      for (int c = 0; c < nch; c += 2) {
        tmem_ld_wait16(ra_);
        if (c + 1 < nch) { issue_chunk(c + 1, rb_); fetch_res(c + 1, qb); }
        finish_chunk(ra_, qa[0], qa[1]);
        if (c + 1 < nch) {
          tmem_ld_wait16(rb_);
          if (c + 2 < nch) { issue_chunk(c + 2, ra_); fetch_res(c + 2, qa); }
          finish_chunk(rb_, qb[0], qb[1]);
        }
      }
      }
      // release the accumulator stage (one arrive per epilogue warp)
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) { if (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]); }
      if (epi_timed) { te2 = clock64(); e_chunks += te2 - te1; }
      if (P.stats_out != nullptr) {
        if (EPI == 2) {
          float a, b, c, d;
          f2_unpack(psum2, a, b); f2_unpack(psq2, c, d);
          psum = a + b; psq = c + d;
        }
        psum = warp_sum(psum);
        psq = warp_sum(psq);
        if (lane == 0) {
          mbar_wait(&stats_empty[acc], acc_phase ^ 1u);
          s_stats[acc * kEpiWarps + ew] = make_float2(psum, psq);
          mbar_arrive(&stats_full[acc]);
        }
        __syncwarp();
      }
      if (epi_timed) e_tail += clock64() - te2;
      if (++acc == P.nacc) { acc = 0; acc_phase ^= 1u; }
    }
    if (epi_timed && ew == 0 && lane == 0) {
      P.dbg_buf[blockIdx.x * 16 + 11] = (unsigned long long)e_pro; P.dbg_buf[blockIdx.x * 16 + 12] = (unsigned long long)e_chunks;
      P.dbg_buf[blockIdx.x * 16 + 13] = (unsigned long long)e_tail;
      P.dbg_buf[blockIdx.x * 16 + 5] = (unsigned long long)epi_wait; P.dbg_buf[blockIdx.x * 16 + 6] = (unsigned long long)(clock64() - epi_begin);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();        // neither CTA retires (or frees tensor memory) while its peer may still signal or read it
  if (warp == 2) {
    tcgen05_fence_after();
    if (CG == 2) tmem_dealloc_2cta(tmem_base, tmem_cols); else tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
// Tuning / profiling knobs.  Production builds have none: every launch parameter is a function of the call's shapes.  Builds
// with -DDS_CONV_DEBUG (tools_dev experiments) read the DS_CONV_* environment variables ONCE, at the first launch.
struct Knobs { int dbg, cg, max_sps, min_stages, sps_cyc, max_stages, generic_epi; };
static const Knobs& knobs() {
  static const Knobs k = [] {
    Knobs v{0, 0, 4, 3, 768, 0, 0};
    const char* e = getenv("DS_CONV_DBG");
    v.dbg = e ? atoi(e) : 0;
#ifdef DS_CONV_DEBUG
    if ((e = getenv("DS_CONV_CG"))) v.cg = atoi(e);
    if ((e = getenv("DS_CONV_MAX_SPS")) && atoi(e) >= 1 && atoi(e) <= 4) v.max_sps = atoi(e);
    if ((e = getenv("DS_CONV_MIN_STAGES"))) v.min_stages = atoi(e);
    if ((e = getenv("DS_CONV_SPS_CYC"))) v.sps_cyc = atoi(e);
    if ((e = getenv("DS_CONV_MAX_STAGES"))) v.max_stages = atoi(e);
    if (getenv("DS_CONV_GENERIC_EPI")) v.generic_epi = 1;
#endif
    return v;
  }();
  return k;
}

static int validate(const ds_conv_gemm_args* a) {
  DS_REQUIRE(a != nullptr, "ds_conv_gemm: null args");
#ifndef DS_CONV_DEBUG
  DS_REQUIRE(knobs().dbg == 0, "ds_conv_gemm: DS_CONV_DBG needs a library built with -DDS_CONV_DEBUG");
#endif
  DS_REQUIRE(a->BK == 32 || a->BK == 64, "ds_conv_gemm: BK must be 32 or 64 (got %d)", a->BK);
  DS_REQUIRE(a->C0 > 0 && a->C0 % a->BK == 0 && a->C1 >= 0 && a->C1 % a->BK == 0,
             "ds_conv_gemm: C0=%d C1=%d must be multiples of BK=%d", a->C0, a->C1, a->BK);
  DS_REQUIRE(a->BN >= 16 && a->BN <= 256 && a->BN % 16 == 0, "ds_conv_gemm: BN=%d must be a multiple of 16 in [16,256]", a->BN);
  DS_REQUIRE(a->Cout_pad % a->BN == 0 && a->Cout <= a->Cout_pad && a->Cout > 0, "ds_conv_gemm: Cout=%d Cout_pad=%d BN=%d", a->Cout, a->Cout_pad, a->BN);
  DS_REQUIRE(a->Hb * a->Wb == BM && a->Hb >= 1 && a->Wb >= 1 && a->Wb <= 256 && a->Hb <= 256, "ds_conv_gemm: tile %dx%d must cover 128 pixels", a->Hb, a->Wb);
  DS_REQUIRE(a->ntaps >= 1 && a->ntaps <= DS_MAX_TAPS && a->groups >= 1 && a->groups <= DS_MAX_GROUPS, "ds_conv_gemm: ntaps=%d groups=%d", a->ntaps, a->groups);
  DS_REQUIRE(a->num_views >= 1 && a->num_views <= 4, "ds_conv_gemm: num_views=%d", a->num_views);
  DS_REQUIRE(a->N > 0 && a->H > 0 && a->W > 0 && a->Hv > 0 && a->Wv > 0, "ds_conv_gemm: bad extents");
  DS_REQUIRE(a->d_src0 && a->d_weight && a->d_e2, "ds_conv_gemm: src0, weight and e2 are required");
  DS_REQUIRE(a->C1 == 0 || a->d_src1, "ds_conv_gemm: C1>0 needs src1");
  DS_REQUIRE(a->ncls == 1 || a->ncls == 9, "ds_conv_gemm: ncls must be 1 or 9");
  DS_REQUIRE(!(a->d_stats_in && !a->d_e1), "ds_conv_gemm: stats_in needs e1");
  DS_REQUIRE(a->d_out || a->d_out_f32_nchw, "ds_conv_gemm: no output");
  DS_REQUIRE(!a->d_out || a->Cout % 16 == 0, "ds_conv_gemm: bf16 output needs Cout %% 16 == 0 (got %d)", a->Cout);
  // the epilogue moves 16 channels (32 bytes) per lane with 256-bit accesses
  DS_REQUIRE(!a->d_out || (reinterpret_cast<uintptr_t>(a->d_out) % 32 == 0 && a->out_sn % 16 == 0 && a->out_sh % 16 == 0 && a->out_sw % 16 == 0),
             "ds_conv_gemm: 16-bit output must be 32-byte aligned with strides that are multiples of 16 elements");
  for (int g = 0; g < a->groups; ++g) DS_REQUIRE(!a->d_out || a->out_goff[g] % 16 == 0, "ds_conv_gemm: out_goff[%d] must be a multiple of 16 elements", g);
  DS_REQUIRE(!a->d_residual || (reinterpret_cast<uintptr_t>(a->d_residual) % 32 == 0 && a->res_sn % 16 == 0 && a->res_sh % 16 == 0 && a->res_sw % 16 == 0),
             "ds_conv_gemm: residual must be 32-byte aligned with strides that are multiples of 16 elements");
  DS_REQUIRE(!(a->per_sample_weights && a->groups != 1), "ds_conv_gemm: per-sample weights with groups");
  for (int g = 0; g < a->groups; ++g)
    for (int t = 0; t < a->ntaps; ++t)
      DS_REQUIRE(a->taps[g][t].view >= 0 && a->taps[g][t].view < a->num_views, "ds_conv_gemm: tap view out of range");
  return DS_OK;
}

static size_t smem_fixed_bytes(const ds_conv_gemm_args* a) {
  const size_t kbt_bytes = (size_t)a->groups * a->ntaps * ((a->C0 + a->C1) / a->BK) * sizeof(int4);     // per-K-block TMA coordinates
  const size_t table_bytes = (size_t)2 * a->ncls * a->Cout_pad * sizeof(float) + kbt_bytes;
  return 1024 + (2 * kMaxStages + 12) * sizeof(uint64_t) + 16 + 2 * kEpiWarps * sizeof(float2) + kEpiWarps * 128 * sizeof(float) + table_bytes + 64;
}
static size_t smem_budget(const ds_conv_gemm_args* a) {
  const size_t f = smem_fixed_bytes(a);
  return f < 226 * 1024 ? 226 * 1024 - f : 0;
}

static void fill_dev(const ds_conv_gemm_args* a, ConvGemmDev& P) {
  memset(&P, 0, sizeof(P));
  P.N = a->N; P.H = a->H; P.W = a->W; P.Hb = a->Hb; P.Wb = a->Wb;
#ifdef DS_CONV_DEBUG
  P.dbg = knobs().dbg;
#else
  P.dbg = 0;        // (ds_conv_gemm refuses DS_CONV_DBG on a build without -DDS_CONV_DEBUG)
#endif
  P.tiles_h = (a->H + a->Hb - 1) / a->Hb;
  P.tiles_w = (a->W + a->Wb - 1) / a->Wb;
  P.tiles_m = P.tiles_h * P.tiles_w;
  // Two-CTA MMA (cta_group::2): the pair computes two M-tiles of one (sample, group, n-tile) with one instruction stream and
  // half of the weight tile per CTA.  It needs an even number of M-tiles; convolutions with enough K per tile to be bound by
  // the MMA issue rate gain from it (ntaps >= 4); DS_CONV_CG=1/2 forces the choice in -DDS_CONV_DEBUG builds.
  {
    const int want = knobs().cg ? knobs().cg : (a->ntaps >= 4 ? 2 : 1);
    const bool even_m = P.tiles_m % 2 == 0;
    const bool flat_ok = a->groups == 1 && !a->per_sample_weights && ((long long)a->N * P.tiles_m) % 2 == 0;
    P.cg = (want == 2 && (even_m || flat_ok) && a->BN % 32 == 0) ? 2 : 1;
    P.pair_flat = (P.cg == 2 && !even_m) ? 1 : 0;
  }
  P.tiles_md = P.pair_flat ? P.tiles_m : P.tiles_m / P.cg;
  P.inv_tiles_md = 1.0f / P.tiles_md;
  P.stage_a_bytes = BM * a->BK * 2;
  P.stage_b_bytes = (a->BN / P.cg) * a->BK * 2;
  P.n_tiles_n = a->Cout_pad / a->BN;
  P.inv_n_tiles_n = 1.0f / P.n_tiles_n; P.inv_tiles_m = 1.0f / P.tiles_m; P.inv_groups = 1.0f / a->groups;
  P.inv_tiles_w = 1.0f / P.tiles_w; P.inv_Wb = 1.0f / P.Wb;
  P.BN = a->BN; P.C0 = a->C0; P.C1 = a->C1;
  P.cblocks0 = a->C0 / a->BK;
  P.cblocks = (a->C0 + a->C1) / a->BK;
  P.ntaps = a->ntaps; P.groups = a->groups; P.per_sample_w = a->per_sample_weights;
  P.src_batch_mod = a->src_batch_mod;
  P.num_kb = P.cblocks * a->ntaps;
  P.num_tiles = (int)((long long)a->N * a->groups * P.tiles_m / P.cg) * P.n_tiles_n;
  P.Cout = a->Cout; P.Cout_pad = a->Cout_pad;
  P.stats_in = reinterpret_cast<const float2*>(a->d_stats_in);
  P.stats_in_slots = a->stats_in_slots; P.out_inv_count = a->stats_out_inv_count; P.eps = a->eps;
  P.e1 = a->d_e1; P.e2 = a->d_e2; P.ncls = a->ncls;
  P.sbias = a->d_sbias; P.sbias_stride = a->sbias_stride; P.act = a->act;
  P.residual = reinterpret_cast<const act_t*>(a->d_residual);
  P.res_sn = a->res_sn; P.res_sh = a->res_sh; P.res_sw = a->res_sw;
  P.out = reinterpret_cast<act_t*>(a->d_out);
  P.out_sn = a->out_sn; P.out_sh = a->out_sh; P.out_sw = a->out_sw;
  for (int g = 0; g < DS_MAX_GROUPS; ++g) P.out_goff[g] = a->out_goff[g];
  P.out_f32 = a->d_out_f32_nchw;
  P.stats_out = reinterpret_cast<float2*>(a->d_stats_out);
  P.stats_slots = a->groups * P.tiles_m * P.n_tiles_n;
  memcpy(P.taps, a->taps, sizeof(P.taps));
}

// Every launch decision of one call: the tile schedule (fill_dev), the epilogue specialisation, the residency (two CTAs per SM),
// the pipeline depth and the grid.  conv_gemm_launch launches exactly this plan and ds_conv_gemm_plan reports it.
struct LaunchPlan { int epi; bool two_per_sm; size_t smem; int grid; };

static int plan_launch(const ds_conv_gemm_args* a, ConvGemmDev& P, LaunchPlan& L) {
  int rc = validate(a);
  if (rc) return rc;
  fill_dev(a, P);
  // epilogue specialisation (see the kernel): the main path needs a 16-bit output whose every chunk is full
  int epi = 0;
  if (a->d_out && !a->d_out_f32_nchw && a->Cout == a->Cout_pad && !(P.dbg & 1) && !knobs().generic_epi) {
    if (a->act == 0) epi = a->d_residual ? 3 : (!a->d_e1 && !a->d_sbias && !a->d_stats_in) ? 4 : 1;
    else if (!a->d_residual && a->d_e1 && a->d_stats_in && !a->d_sbias) epi = 2;      // ConvNeXt conv1: fold + GELU, no per-sample bias
  }
  // two resident CTAs per SM for the plain 1x1 convolutions whose accumulator pair fits half of the tensor memory (see the kernel)
  // (BN <= 128: each CTA keeps its double-buffered accumulator in half of the tensor memory; BN <= 256: a single accumulator per CTA,
  // the other CTA's work covers the wait between a tile's MMAs and its epilogue)
  const size_t fixed_bytes = smem_fixed_bytes(a);
  const size_t half_budget = fixed_bytes < 111 * 1024 ? 111 * 1024 - fixed_bytes : 0;
  const bool two_per_sm = epi == 4 && P.cg == 1 && a->ntaps == 1 && half_budget >= 2 * ((size_t)P.stage_a_bytes + P.stage_b_bytes);
  P.nacc = (two_per_sm && 2 * a->BN > 256) ? 1 : 2;
  const size_t budget = two_per_sm ? half_budget : smem_budget(a);
  // K-blocks per stage: one barrier round trip per stage costs a few hundred cycles on the single MMA-issuing thread, so every
  // stage should carry >= ~384 cycles of tensor work (BK/16 MMAs of BN/2 cycles each per K-block) while >= 4 stages still fit.
  P.sps = 1;
  {
    const size_t sub = (size_t)P.stage_a_bytes + P.stage_b_bytes;
    const int cyc = (a->BK / 16) * (a->BN / 2);
    const int max_sps = two_per_sm ? 1 : knobs().max_sps;          // 4: the producer keeps at most 4 table entries in registers
    const int min_stages = knobs().min_stages;    // 3: three stages already saturate the pipeline (measured); deeper rings buy nothing
    const int cyc_target = knobs().sps_cyc;       // 768: measured, two barrier round trips per ~768 MMA cycles keep the single issuing thread off the critical path
    while (P.sps < max_sps && P.sps * cyc < cyc_target && P.sps < P.num_kb && (size_t)(P.sps + 1) * sub * min_stages <= budget) ++P.sps;
  }
  const size_t stage_bytes = (size_t)P.sps * ((size_t)P.stage_a_bytes + P.stage_b_bytes);
  int stages = (int)(budget / stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (knobs().max_stages >= 2 && knobs().max_stages < stages) stages = knobs().max_stages;      // (-DDS_CONV_DEBUG experiment knob)
  // (the ring spans tiles of the persistent loop: small-K convs prefetch several tiles ahead, so it is never clamped to K)
  DS_REQUIRE(stages >= 2, "ds_conv_gemm: epilogue tables leave no room for a 2-stage pipeline (Cout_pad=%d ncls=%d)", a->Cout_pad, a->ncls);
  P.stages = stages;
  L.epi = epi;
  L.two_per_sm = two_per_sm;
  L.smem = fixed_bytes + stages * stage_bytes;
  const int slots = two_per_sm ? 2 * num_sms() : num_sms();
  L.grid = P.num_tiles < slots ? P.num_tiles : slots;
  if (P.cg == 2) { const int pairs = num_sms() / 2; L.grid = 2 * (P.num_tiles < pairs ? P.num_tiles : pairs); }
  return DS_OK;
}

static int conv_gemm_launch(const ds_conv_gemm_args* a, cudaStream_t stream) {
  ConvGemmDev P;
  LaunchPlan L;
  int rc = plan_launch(a, P, L);
  if (rc) return rc;
  EncodeTiledFn encode = get_encode_fn();
  DS_REQUIRE(encode != nullptr, "ds_conv_gemm: cuTensorMapEncodeTiled entry point not available");

  TmaMaps maps;          // per call (host threads may launch concurrently); unused slots are copies of a valid map (prefetch-safe)
  const CUtensorMapSwizzle swz = a->BK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;

  for (int s = 0; s < 2; ++s) {
    const int C = s == 0 ? a->C0 : a->C1;
    const char* base = reinterpret_cast<const char*>(s == 0 ? a->d_src0 : a->d_src1);
    for (int v = 0; v < 4; ++v) {
      if (C == 0 || v >= a->num_views) { maps.a[s][v] = maps.a[0][0]; continue; }
      const int Wv = a->view_wv[v] > 0 ? a->view_wv[v] : a->Wv, Hv = a->view_hv[v] > 0 ? a->view_hv[v] : a->Hv;
      cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)Wv, (cuuint64_t)Hv,
                            (cuuint64_t)((s == 0 && a->src_batch_mod > 0) ? a->src_batch_mod : a->N)};
      cuuint64_t strides[3] = {(cuuint64_t)a->view_sw * C * 2, (cuuint64_t)a->view_sh * C * 2, (cuuint64_t)a->view_sn * C * 2};
      cuuint32_t box[4] = {(cuuint32_t)a->BK, (cuuint32_t)a->Wb, (cuuint32_t)a->Hb, 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      void* gaddr = const_cast<char*>(base) + (size_t)a->view_off[v] * C * 2;
      CUresult r = encode(&maps.a[s][v], (kOperandIsFp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), 4, gaddr, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      DS_REQUIRE(r == CUDA_SUCCESS, "ds_conv_gemm: cuTensorMapEncodeTiled(A src %d view %d) failed with %d (C=%d Wv=%d Hv=%d)", s, v, (int)r, C, Wv, Hv);
    }
  }
  {
    const long long K = (long long)a->ntaps * (a->C0 + a->C1);
    const int Z = a->per_sample_weights ? a->N : a->groups;
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)a->Cout_pad, (cuuint64_t)Z};
    cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)K * 2 * a->Cout_pad};
    cuuint32_t box[3] = {(cuuint32_t)a->BK, (cuuint32_t)(a->BN / P.cg), 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode(&maps.b, (kOperandIsFp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), 3, const_cast<void*>(a->d_weight), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DS_REQUIRE(r == CUDA_SUCCESS, "ds_conv_gemm: cuTensorMapEncodeTiled(B) failed with %d (K=%lld Cout_pad=%d)", (int)r, K, a->Cout_pad);
  }

  const int epi = L.epi, grid = L.grid;
  const size_t smem = L.smem;
  static unsigned long long* dbg_buf = nullptr;
  P.dbg_buf = nullptr;
  if (P.dbg & 64) {
    if (!dbg_buf) DS_CHECK_CUDA(cudaMalloc(&dbg_buf, sizeof(unsigned long long) * 16 * 1024));
    DS_CHECK_CUDA(cudaMemsetAsync(dbg_buf, 0, sizeof(unsigned long long) * 16 * 1024, stream));
    P.dbg_buf = dbg_buf;
  }
#define DS_LAUNCH_CONV(BKV, CGV, EPIV)                                                                                                \
  do {                                                                                                                                \
    DS_CHECK_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<BKV, CGV, EPIV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    cudaLaunchConfig_t cfg;                                                                                                           \
    memset(&cfg, 0, sizeof(cfg));                                                                                                     \
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kNumThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;                    \
    cudaLaunchAttribute attr[2];                                                                                                      \
    int na = 0;                                                                                                                       \
    if (CGV == 2) {                                                                                                                   \
      attr[na].id = cudaLaunchAttributeClusterDimension;                                                                              \
      attr[na].val.clusterDim.x = CGV; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;                                 \
      ++na;                                                                                                                           \
    }                                                                                                                                 \
    if (pdl_enabled()) {                                                                                                              \
      attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                                               \
      attr[na].val.programmaticStreamSerializationAllowed = 1;                                                                        \
      ++na;                                                                                                                           \
    }                                                                                                                                 \
    cfg.attrs = attr; cfg.numAttrs = na;                                                                                              \
    DS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_gemm_kernel<BKV, CGV, EPIV>, maps, P));                                               \
  } while (0)
#define DS_LAUNCH_CONV_E(BKV, CGV)                                                                                  \
  do {                                                                                                              \
    if (epi == 1) DS_LAUNCH_CONV(BKV, CGV, 1); else if (epi == 2) DS_LAUNCH_CONV(BKV, CGV, 2);                     \
    else if (epi == 3) DS_LAUNCH_CONV(BKV, CGV, 3); else if (epi == 4) DS_LAUNCH_CONV(BKV, CGV, 4);                \
    else DS_LAUNCH_CONV(BKV, CGV, 0);                                                                              \
  } while (0)
  if (a->BK == 64) { if (P.cg == 2) DS_LAUNCH_CONV_E(64, 2); else DS_LAUNCH_CONV_E(64, 1); }
  else             { if (P.cg == 2) DS_LAUNCH_CONV_E(32, 2); else DS_LAUNCH_CONV_E(32, 1); }
#undef DS_LAUNCH_CONV_E
#undef DS_LAUNCH_CONV
  DS_CHECK_CUDA(cudaGetLastError());
  if (P.dbg & 64) {      // profiling only: where each role of the CTA spent its cycles (mean over CTAs)
    static unsigned long long host[16 * 1024];
    DS_CHECK_CUDA(cudaStreamSynchronize(stream));
    DS_CHECK_CUDA(cudaMemcpy(host, dbg_buf, sizeof(unsigned long long) * 16 * grid, cudaMemcpyDeviceToHost));
    double m[16] = {0};
    for (int b = 0; b < grid; ++b) for (int i = 0; i < 16; ++i) m[i] += (double)host[b * 16 + i] / grid;
    fprintf(stderr, "[conv dbg] cg %d tiles/cta %.1f kb/tile %d sps %d stages %d | producer: wait_empty %.0f of %.0f | mma: wait_full %.0f wait_tmem_empty %.0f of %.0f | epilogue(w4): wait_tmem_full %.0f of %.0f cycles | mma detail: fence %.0f issue %.0f commit %.0f | epi detail: prologue %.0f chunks %.0f tail %.0f\n",
            P.cg, (double)P.num_tiles * P.cg / grid, P.num_kb, P.sps, P.stages, m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[8], m[9], m[10], m[11], m[12], m[13]);
  }
  return DS_OK;
}

// ---------------------------------------------------------------------------------------------
// CUDA-core cross-check of the same contract (tests only): one thread per (pixel, out channel).
// ---------------------------------------------------------------------------------------------
__global__ void conv_gemm_ref_kernel(const ConvGemmDev P, const act_t* src0, const act_t* src1,
                                     const act_t* weight, long long view_sn, long long view_sh,
                                     long long view_sw, const long long* view_off_dev /* [4] offsets, [4] widths, [4] heights */) {
  const long long total = (long long)P.N * P.groups * P.H * P.W * P.Cout;
  const long long K = (long long)P.ntaps * (P.C0 + P.C1);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int o = (int)(i % P.Cout);
    long long r = i / P.Cout;
    int w = (int)(r % P.W); r /= P.W;
    int h = (int)(r % P.H); r /= P.H;
    int g = (int)(r % P.groups);
    int n = (int)(r / P.groups);
    const int nsrc = P.src_batch_mod > 0 ? (n % P.src_batch_mod) : n;
    const act_t* wrow = weight + ((long long)(P.per_sample_w ? n : g) * P.Cout_pad + o) * K;
    float acc = 0.f;
    for (int t = 0; t < P.ntaps; ++t) {
      const ds_conv_tap tp = P.taps[g][t];
      const int y = h + tp.dy, x = w + tp.dx;
      if (y < 0 || y >= view_off_dev[8 + tp.view] || x < 0 || x >= view_off_dev[4 + tp.view]) continue;
      const long long pix0 = view_off_dev[tp.view] + nsrc * view_sn + y * view_sh + x * view_sw;     // source 0: batch modulus
      const long long pix1 = view_off_dev[tp.view] + n * view_sn + y * view_sh + x * view_sw;
      for (int c = 0; c < P.C0 + P.C1; ++c) {
        const float a = c < P.C0 ? act2f(src0[pix0 * P.C0 + c]) : act2f(src1[pix1 * P.C1 + (c - P.C0)]);
        acc = fmaf(a, act2f(wrow[(long long)t * (P.C0 + P.C1) + c]), acc);
      }
    }
    float mean = 0.f, rstd = 1.f;
    if (P.stats_in) { const float2 mr = *stats_sample(P.stats_in, P.stats_in_slots, nsrc); mean = mr.x; rstd = mr.y; }
    int cls = 0;
    if (P.ncls == 9) cls = (h == 0 ? 0 : (h == P.H - 1 ? 2 : 1)) * 3 + (w == 0 ? 0 : (w == P.W - 1 ? 2 : 1));
    float v = acc * rstd + P.e2[(size_t)cls * P.Cout_pad + o];
    if (P.e1) v = fmaf(-mean * rstd, P.e1[(size_t)cls * P.Cout_pad + o], v);
    if (P.sbias) v += P.sbias[(size_t)n * P.sbias_stride + o];
    if (P.act == 1) v = gelu_erf(v);   // exact erf here: cross-checks the fast form used by the tcgen05 epilogue
    if (P.residual) v += act2f(P.residual[n * P.res_sn + h * P.res_sh + w * P.res_sw + o]);
    if (P.out) P.out[P.out_goff[g] + n * P.out_sn + h * P.out_sh + w * P.out_sw + o] = f2act(v);
    if (P.out_f32) P.out_f32[(((size_t)n * P.Cout + o) * P.H + h) * P.W + w] = v;
  }
}

static int conv_gemm_reference_launch(const ds_conv_gemm_args* a, cudaStream_t stream) {
  int rc = validate(a);
  if (rc) return rc;
  ConvGemmDev P;
  fill_dev(a, P);
  long long* voff = nullptr;
  long long vtab[12];      // (pageable host source: the copy is staged before cudaMemcpyAsync returns)
  for (int v = 0; v < 4; ++v) {
    vtab[v] = a->view_off[v];
    vtab[4 + v] = a->view_wv[v] > 0 ? a->view_wv[v] : a->Wv;
    vtab[8 + v] = a->view_hv[v] > 0 ? a->view_hv[v] : a->Hv;
  }
  DS_CHECK_CUDA(cudaMallocAsync(&voff, sizeof(vtab), stream));
  DS_CHECK_CUDA(cudaMemcpyAsync(voff, vtab, sizeof(vtab), cudaMemcpyHostToDevice, stream));
  conv_gemm_ref_kernel<<<num_sms() * 8, 256, 0, stream>>>(P, reinterpret_cast<const act_t*>(a->d_src0),
                                                          reinterpret_cast<const act_t*>(a->d_src1),
                                                          reinterpret_cast<const act_t*>(a->d_weight),
                                                          a->view_sn, a->view_sh, a->view_sw, voff);
  DS_CHECK_CUDA(cudaGetLastError());
  DS_CHECK_CUDA(cudaFreeAsync(voff, stream));
  return DS_OK;
}

}  // namespace ds

extern "C" int ds_conv_gemm(const ds_conv_gemm_args* args, void* stream) {
  return ds::conv_gemm_launch(args, reinterpret_cast<cudaStream_t>(stream));
}
extern "C" int ds_conv_gemm_reference(const ds_conv_gemm_args* args, void* stream) {
  return ds::conv_gemm_reference_launch(args, reinterpret_cast<cudaStream_t>(stream));
}
extern "C" int ds_conv_gemm_plan(const ds_conv_gemm_args* a, ds_conv_gemm_plan_info* info) {
  DS_REQUIRE(info != nullptr, "ds_conv_gemm_plan: null info");
  ds::ConvGemmDev P;
  ds::LaunchPlan L;
  const int rc = ds::plan_launch(a, P, L);
  if (rc) return rc;
  info->BK = a->BK; info->BN = a->BN; info->cg = P.cg; info->pair_flat = P.pair_flat; info->epi = L.epi;
  info->two_per_sm = L.two_per_sm ? 1 : 0; info->nacc = P.nacc; info->sps = P.sps; info->stages = P.stages;
  info->num_tiles = P.num_tiles; info->grid = L.grid;
  return ds::DS_OK;
}
extern "C" int ds_conv_gemm_stats_slots(const ds_conv_gemm_args* a) {
  if (!a || a->Hb <= 0 || a->Wb <= 0 || a->BN <= 0) return -1;
  ds::ConvGemmDev P;
  ds::fill_dev(a, P);
  return P.stats_slots;
}
