// Fused  PreNorm -> to_qkv -> (softmax_d(q) * scale,  online softmax_n(k),  partial context  S = P^T V)  for the U-Net's
// LinearCrossAttentionAdd / LinearCrossAttention (model/diffusion_components.py:148-151,263,271-289 and :171-207):
// the 1x1 to_qkv convolution runs on tcgen05 (TMA-fed, TMEM accumulator 128 pixels x 192 channels of a head pair) and its epilogue keeps k
// and v on chip -- they are never written to HBM: per 128-pixel tile the epilogue turns k into P = exp(k - m[d]) (softmax over n is
// shift invariant per row, so any m[d] common to the pixels of a partial is exact), stages P and V as bf16 in shared
// memory and contracts them over the pixels with warp-level MMAs into S[d][e] (+ Z[d] = sum_n P through a column of ones);
// q is soft-maxed over its 32 head channels in registers and written as the only per-pixel output (q').
// The stabiliser is chosen per row d of the partial (see the epilogue), so no row can lose all of its pixels to underflow and no
// later tile can overflow P.
// One partial (S[32][32], Z[32], m[32]) per (sample, head, 512-pixel chunk) leaves the kernel in the format
// attn_reduce_kernel / attn_fold_kernel already consume (ds_attn_finalize).  Replaces a to_qkv launch (which wrote 384
// channels per pixel) and an attn_ctx_partial launch (which read them back).
//
// CTA = 8 warps, two CTAs per SM, persistent over (sample, chunk, head pair) items:  warp 0 activation TMA producer, warp 1 MMA
// issuer, warp 2 TMEM allocator + weight TMA producer, warps 4-7 epilogue (thread = pixel row, the pair's q, k and v; for the context
// MMAs warp w owns head w/2 of the pair, d rows 16*(w%2)..+15).
#include "common.cuh"
#include "../../include/diffusynth_b200.h"
#include "umma.cuh"

namespace ds {

// Work item = (sample, 512-pixel chunk, head pair): the GEMM of an item is 128 pixels x 192 channels (q | k | v of two heads), so the
// accumulator needs 192 of the 512 tensor-memory columns and a CTA 99 KB of shared memory: TWO CTAs live on an SM and interleave --
// while one waits for its accumulator, its exponentials (MUFU) or a block barrier, the other one runs.  The activation tile is read
// twice (once per head pair; the pair's items are adjacent in the work order, the second read hits L2).
static constexpr int AQ_THREADS = 256;                    // warps 0-2: roles (3 idle), warps 4-7: epilogue
static constexpr int AQ_BK = 32;                          // channels per K-block (64-byte rows, SWIZZLE_64B): divides every C
static constexpr int AQ_STAGES = 3;
static constexpr int AQ_HID = 128, AQ_HEADS = 4, AQ_DH = 32, AQ_NOUT = 3 * AQ_HID;
static constexpr int AQ_PN = 3 * 2 * AQ_DH;               // 192 GEMM columns of a head pair: q [0,64) | k [64,128) | v [128,192)
static constexpr int AQ_TILE = 128;                       // pixels per MMA tile
static constexpr int AQ_SUB = 4;                          // tiles per chunk (one partial per 512 pixels, as ds_attn_chunks)
static constexpr int AQ_A_BYTES = AQ_TILE * AQ_BK * 2;    // 8 KB
static constexpr int AQ_B_BYTES = AQ_PN * AQ_BK * 2;      // 12 KB
static constexpr int AQ_STAGE_BYTES = AQ_A_BYTES + AQ_B_BYTES;
static constexpr int AQ_PITCH = 2 * 2 * AQ_DH + 16;       // bytes per staged P / V row (2 heads): 8 rows x 16 B hit 8 different bank groups
static constexpr int AQ_PART = AQ_DH * AQ_DH + 2 * AQ_DH;
static constexpr int AQ_SMEM = 1024 + AQ_STAGES * AQ_STAGE_BYTES + 2 * AQ_TILE * AQ_PITCH + AQ_PN * 4 + 256 + 7 * 2 * AQ_DH * 4;
// Stabiliser bounds (log2 units, see the epilogue).  A row whose first-tile maximum lies more than AQ_ROW_LOW below its head's
// takes its own stabiliser: under the head's, its largest P would be < 2^-100 and all of them could flush to 0 (ex2.approx.ftz
// ends at 2^-126).  A later tile in which some P would exceed 2^AQ_RESCALE raises the stabiliser and rescales S and Z: P <= 2^96,
// 512 of them times |v| < 2^22 stay inside fp32 / bf16.
static constexpr float AQ_ROW_LOW = 100.f;
static constexpr float AQ_RESCALE = 96.f;

struct AttnQkvDev {
  int N, npix, C, num_kb, x_batch_mod, chunks, items;
  const float2* stats_in; int stats_in_slots;
  const float* e1; const float* e2; const float* sbias; long long sbias_stride;
  act_t* qout; float* part; float scale;
};

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
// q' in [0, scale]: one F2FP (pack16's clamp to the finite fp16 range costs two FMNMX per value)
__device__ __forceinline__ uint32_t pack_q(float lo, float hi) {
#ifdef DS_OPERANDS_BF16
  return pack16(lo, hi);
#else
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
#endif
}
// Column maxima of a warp's 32 x 32 block (lane = pixel row, k[j] = column j): a butterfly that halves the columns a lane keeps at
// every step (16 + 8 + 4 + 2 + 1 shuffles); lane l returns the maximum of column l over the lanes with `valid`.
__device__ __forceinline__ float col_max32(const uint32_t (&k)[32], bool valid, int lane) {
  float t[16];
  const bool up16 = (lane & 16) != 0;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float lo = valid ? __uint_as_float(k[j]) : -INFINITY, hi = valid ? __uint_as_float(k[j + 16]) : -INFINITY;
    t[j] = fmaxf(up16 ? hi : lo, __shfl_xor_sync(0xffffffffu, up16 ? lo : hi, 16));
  }
#pragma unroll
  for (int s = 8; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int j = 0; j < s; ++j) t[j] = fmaxf(up ? t[j + s] : t[j], __shfl_xor_sync(0xffffffffu, up ? t[j] : t[j + s], s));
  }
  return t[0];
}
// named barrier that also returns whether any participating thread passed `v`
__device__ __forceinline__ bool bar_red_or(int id, int nthreads, bool v) {
  uint32_t r;
  asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
               : "=r"(r) : "r"((uint32_t)v), "r"(id), "r"(nthreads) : "memory");
  return r != 0;
}
__device__ __forceinline__ void sts_128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__global__ void __launch_bounds__(AQ_THREADS, 2)
attn_qkv_ctx_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ AttnQkvDev P) {
  extern __shared__ __align__(1024) uint8_t aq_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(aq_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_p = smem + AQ_STAGES * AQ_STAGE_BYTES;                        // [128][AQ_PITCH] bf16 P rows (2 heads)
  uint8_t* s_v = s_p + AQ_TILE * AQ_PITCH;                                 // [128][AQ_PITCH] bf16 V rows
  float* s_t = reinterpret_cast<float*>(s_v + AQ_TILE * AQ_PITCH);         // [192] per-sample additive constants of the fold
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_t + AQ_PN);
  uint64_t* empty_bar = full_bar + AQ_STAGES;
  // one accumulator (192 columns): the epilogue pulls it into registers piece by piece and releases it before the context MMAs
  uint64_t* tmem_full = empty_bar + AQ_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  // stabiliser of the item's 64 k rows (2 heads x 32 d, log2 units): column maxima per epilogue warp, m, -mb, and a rescale step
  float* s_red = reinterpret_cast<float*>(tmem_base_smem + 4);             // [4 lane groups][64] (16-byte aligned: s_nm / s_dl are read as float4)
  float* s_m = s_red + 4 * 2 * AQ_DH;                                      // [64] m[d]
  float* s_nm = s_m + 2 * AQ_DH;                                           // [64] -mb[d]  (P = exp2(rl2 acc + s_nm), m = mb + tk)
  float* s_dl = s_nm + 2 * AQ_DH;                                          // [64] increase of m in a rescaling tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { prefetch_tmap(&map_a); prefetch_tmap(&map_b); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < AQ_STAGES; ++s) { mbar_init(&full_bar[s], 2); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) umma::tmem_alloc(tmem_base_smem, 256);
  pdl_launch_dependents();
  pdl_wait();
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  auto tiles_of = [&](int chunk) { const int left = P.npix - chunk * AQ_SUB * AQ_TILE; const int t = (left + AQ_TILE - 1) / AQ_TILE; return t < AQ_SUB ? t : AQ_SUB; };
  // item -> (sample, chunk, head pair); the two head pairs of a (sample, chunk) are neighbours in the work order
  auto decode = [&](int item, int& n, int& chunk, int& hp) { hp = item & 1; const int r = item >> 1; n = r / P.chunks; chunk = r - n * P.chunks; };

  if (warp == 0) {
    // ================= activation producer =================
    int stage = 0; uint32_t phase = 0;
    for (int item = blockIdx.x; item < P.items; item += gridDim.x) {
      int n, chunk, hp;
      decode(item, n, chunk, hp);
      const int nsrc = P.x_batch_mod > 0 ? n % P.x_batch_mod : n;
      const int nt = tiles_of(chunk);
      for (int sub = 0; sub < nt; ++sub) {
        const int p0 = (chunk * AQ_SUB + sub) * AQ_TILE;
        for (int kb = 0; kb < P.num_kb; ++kb) {
          mbar_wait_warp(&empty_bar[stage], phase ^ 1u);
          if (umma::elect_one()) {
            mbar_expect_tx(&full_bar[stage], AQ_A_BYTES);
            tma_load_3d(smem + stage * AQ_STAGE_BYTES, &map_a, &full_bar[stage], kb * AQ_BK, p0, nsrc);
          }
          __syncwarp();
          if (++stage == AQ_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 2) {
    // ================= weight producer (the pair's 192 rows of the 384 x C matrix stream once per tile; L2 resident) =================
    int stage = 0; uint32_t phase = 0;
    for (int item = blockIdx.x; item < P.items; item += gridDim.x) {
      int n, chunk, hp;
      decode(item, n, chunk, hp);
      const int nt = tiles_of(chunk);
      for (int sub = 0; sub < nt; ++sub) {
        for (int kb = 0; kb < P.num_kb; ++kb) {
          mbar_wait_warp(&empty_bar[stage], phase ^ 1u);
          if (umma::elect_one()) {
            uint8_t* sb = smem + stage * AQ_STAGE_BYTES + AQ_A_BYTES;
            mbar_expect_tx(&full_bar[stage], AQ_B_BYTES);
#pragma unroll
            for (int j = 0; j < 3; ++j) tma_load_3d(sb + j * (AQ_B_BYTES / 3), &map_b, &full_bar[stage], kb * AQ_BK, j * AQ_HID + hp * 2 * AQ_DH, 0);
          }
          __syncwarp();
          if (++stage == AQ_STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: D[128 x 192] = X[128 x C] W_pair^T, one N = 192 instruction per K step =================
    const uint32_t idesc = umma::idesc_f16(128, AQ_PN);
    int stage = 0; uint32_t phase = 0, acc_phase = 0;
    for (int item = blockIdx.x; item < P.items; item += gridDim.x) {
      int n, chunk, hp;
      decode(item, n, chunk, hp);
      const int nt = tiles_of(chunk);
      for (int sub = 0; sub < nt; ++sub) {
        mbar_wait_warp(tmem_empty, acc_phase ^ 1u);
        umma::fence_after();
        for (int kb = 0; kb < P.num_kb; ++kb) {
          mbar_wait_warp(&full_bar[stage], phase);
          umma::fence_after();
          if (umma::elect_one()) {
            const uint32_t sa = smem_u32(smem + stage * AQ_STAGE_BYTES);
            const uint64_t adesc = umma::kmajor_desc<AQ_BK>(sa);
            const uint64_t bdesc = umma::kmajor_desc<AQ_BK>(sa + AQ_A_BYTES);
#pragma unroll
            for (int k = 0; k < AQ_BK / 16; ++k)
              umma::mma_f16(tmem_base, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
            umma::commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == AQ_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (umma::elect_one()) umma::commit(tmem_full);
        __syncwarp();
        acc_phase ^= 1u;
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: thread = pixel row (TMEM lane), all 192 columns of the pair =================
    const int ew = warp - 4;                                    // = TMEM lane group
    const int row = ew * 32 + lane;
    const int etid = ew * 32 + lane;
    const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16);
    const int hl = ew >> 1, mt = ew & 1;                        // context MMAs: head of the pair, 16-row half of d
    const uint32_t sp_row = smem_u32(s_p) + (uint32_t)(row * AQ_PITCH), sv_row = smem_u32(s_v) + (uint32_t)(row * AQ_PITCH);
    const int lr = lane & 7, lmat = lane >> 3;
    uint32_t acc_phase = 0;
    constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;
    const uint32_t tq_s = smem_u32(s_t), tv_s = smem_u32(s_t + 4 * AQ_DH);
    // (volatile on purpose: letting the compiler batch these loads costs registers and spills)
    auto lds4 = [](uint32_t addr) { float4 v; asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory"); return v; };

    for (int item = blockIdx.x; item < P.items; item += gridDim.x) {
      int n, chunk, hp;
      decode(item, n, chunk, hp);
      const int nsrc = P.x_batch_mod > 0 ? n % P.x_batch_mod : n;
      float mean = 0.f, rstd = 1.f;
      if (P.stats_in != nullptr) { const float2 mr = __ldg(stats_sample(P.stats_in, P.stats_in_slots, nsrc)); mean = mr.x; rstd = mr.y; }
      const float rl2 = rstd * kLog2e;
      // additive constants of the GroupNorm fold + bias for this sample: value = rstd * acc + t[col]; q and k work in the log2
      // domain (their only consumers are exponentials): value * log2(e) = (rstd log2 e) * acc + t[col] log2 e
      for (int l = etid; l < AQ_PN; l += 128) {
        const int col = (l >> 6) * AQ_HID + hp * 2 * AQ_DH + (l & 63);
        float t = __ldg(P.e2 + col);
        if (P.e1 != nullptr) t = fmaf(-mean * rstd, __ldg(P.e1 + col), t);
        if (P.sbias != nullptr) t += __ldg(P.sbias + (size_t)n * P.sbias_stride + col);
        s_t[l] = l < 4 * AQ_DH ? t * kLog2e : t;
      }
      // Stabiliser of the exponentials, one per row d of the partial (log2 domain, of the bare product rl2 acc; the per-row constant
      // tk[d] -- bias, label key, GroupNorm mean fold -- never enters the exponent and is reported through m).  Soft-max over n is
      // shift invariant per row, so any value that is the same for every pixel of the partial is exact.  A row takes its head's
      // maximum over the valid pixels of the item's first tile, mh, unless its own first-tile maximum r[d] lies more than AQ_ROW_LOW
      // below mh (a block input with a large mean-to-std ratio spreads the rows of a head apart by rl2 mean sum_c W'[d,c]); such a
      // row takes r[d], so its largest pixel gives P = 1 and Z[d] >= 1.  Rows within range keep exactly the head value, so their
      // P, S, Z and m are bit-identical to a per-head stabiliser.  A later tile in which some P would exceed 2^AQ_RESCALE raises
      // the row's stabiliser to that tile's maximum and rescales S and Z, as attn_ctx_partial_kernel does.
      float c[4][4], cz[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { cz[i] = 0.f; for (int j = 0; j < 4; ++j) c[i][j] = 0.f; }
      umma::named_bar_sync(2, 128);                              // s_t visible; the previous item's staging reads are done
      const uint32_t nm_s = smem_u32(s_nm), dl_s = smem_u32(s_dl);

      const int nt = tiles_of(chunk);
      for (int sub = 0; sub < nt; ++sub) {
        const int p0 = (chunk * AQ_SUB + sub) * AQ_TILE;
        const bool valid = p0 + row < P.npix;                    // (false only in the ragged last tile of a sample)
        mbar_wait_warp(tmem_full, acc_phase);
        umma::fence_after();
        // ---- k (columns 64..127) -> P = exp2(rl2 acc - mb[d]) as bf16 rows ----
        bool rescale;
        {
          uint32_t k0[32], k1[32];
          umma::ld_32x32b_x32(t_row + 64u, k0);
          umma::ld_32x32b_x32(t_row + 96u, k1);
          umma::ld_wait32(k0);
          umma::ld_wait32(k1);
          if (sub == 0) {
            // first tile: row maxima r[d] of acc (rl2 > 0: max(rl2 acc) = rl2 max(acc)); warps 4 and 5 (etid < 64) hold head 0 and
            // head 1 of the pair, lane = d, so the head maximum is a warp maximum
            const float r0 = col_max32(k0, valid, lane), r1 = col_max32(k1, valid, lane);
            s_red[ew * 64 + lane] = r0;
            s_red[ew * 64 + 32 + lane] = r1;
            umma::named_bar_sync(1, 128);
            if (etid < 2 * AQ_DH) {
              const float mx = fmaxf(fmaxf(s_red[etid], s_red[64 + etid]), fmaxf(s_red[128 + etid], s_red[192 + etid]));
              const float mh = rl2 * warp_max(mx), mr = rl2 * mx;
              const float mb = mr < mh - AQ_ROW_LOW ? mr : mh;
              s_m[etid] = mb + s_t[2 * AQ_DH + etid];               // m[d] = mb[d] + tk[d]
              s_nm[etid] = -mb;
              s_dl[etid] = 0.f;
            }
            umma::named_bar_sync(1, 128);
          }
          // e = rl2 acc - mb in place (log2 of P), and this pixel's largest e
          float emax = -INFINITY;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 a = lds4(nm_s + (uint32_t)(hh * 32 + 4 * j4) * 4u);
              const float na[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                uint32_t& r = hh == 0 ? k0[4 * j4 + i] : k1[4 * j4 + i];
                const float e = fmaf(__uint_as_float(r), rl2, na[i]);
                emax = fmaxf(emax, e);
                r = __float_as_uint(e);
              }
            }
          }
          rescale = sub > 0 && bar_red_or(1, 128, valid && emax > AQ_RESCALE);
          if (rescale) {
            // rare: some row of this tile rose more than AQ_RESCALE above its stabiliser -> raise m[d] by the tile's excess
            // max(0, max_pix e[d]): the maximum of positive floats is the maximum of their bit patterns (s_dl is 0 here)
            if (valid) {
#pragma unroll
              for (int j = 0; j < 64; ++j) {
                const float e = __uint_as_float(j < 32 ? k0[j] : k1[j - 32]);
                if (e > 0.f) atomicMax(reinterpret_cast<int*>(s_dl) + j, __float_as_int(e));
              }
            }
            umma::named_bar_sync(1, 128);
            if (etid < 2 * AQ_DH) {
              const float dl = s_dl[etid];
              s_m[etid] += dl;
              s_nm[etid] -= dl;
            }
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                const float4 a = lds4(dl_s + (uint32_t)(hh * 32 + 4 * j4) * 4u);
                const float da[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  uint32_t& r = hh == 0 ? k0[4 * j4 + i] : k1[4 * j4 + i];
                  r = __float_as_uint(__uint_as_float(r) - da[i]);
                }
              }
            }
            // S and Z so far were taken against the old m: rows d = 16 mt + g and + 8 of head hl (this thread's accumulators)
            const int g = lane >> 2;
            float sl, sh;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sl) : "f"(-s_dl[hl * AQ_DH + mt * 16 + g]));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(sh) : "f"(-s_dl[hl * AQ_DH + mt * 16 + g + 8]));
#pragma unroll
            for (int i = 0; i < 4; ++i) { c[i][0] *= sl; c[i][1] *= sl; c[i][2] *= sh; c[i][3] *= sh; }
            cz[0] *= sl; cz[1] *= sl; cz[2] *= sh; cz[3] *= sh;
          }
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
            for (int q8 = 0; q8 < 4; ++q8) {
              uint32_t o[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t r0 = hh == 0 ? k0[q8 * 8 + 2 * j] : k1[q8 * 8 + 2 * j], r1 = hh == 0 ? k0[q8 * 8 + 2 * j + 1] : k1[q8 * 8 + 2 * j + 1];
                float e0, e1;
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(__uint_as_float(r0)));
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(__uint_as_float(r1)));
                o[j] = valid ? pack_bf16(e0, e1) : 0u;
              }
              sts_128(sp_row + (uint32_t)(hh * 64 + q8 * 16), o[0], o[1], o[2], o[3]);
            }
          }
        }
        // ---- v (columns 128..191) as bf16 rows ----
        {
          uint32_t v0[32], v1[32];
          umma::ld_32x32b_x32(t_row + 128u, v0);
          umma::ld_32x32b_x32(t_row + 160u, v1);
          umma::ld_wait32(v0);
          umma::ld_wait32(v1);
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
            for (int q8 = 0; q8 < 4; ++q8) {
              uint32_t o[4];
              const float4 ta = lds4(tv_s + (uint32_t)(hh * 32 + q8 * 8) * 4u), tb = lds4(tv_s + (uint32_t)(hh * 32 + q8 * 8 + 4) * 4u);
              const float tvv[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t r0 = hh == 0 ? v0[q8 * 8 + 2 * j] : v1[q8 * 8 + 2 * j], r1 = hh == 0 ? v0[q8 * 8 + 2 * j + 1] : v1[q8 * 8 + 2 * j + 1];
                o[j] = pack_bf16(fmaf(__uint_as_float(r0), rstd, tvv[2 * j]), fmaf(__uint_as_float(r1), rstd, tvv[2 * j + 1]));      // (rows past the end of the sample meet P = 0)
              }
              sts_128(sv_row + (uint32_t)(hh * 64 + q8 * 16), o[0], o[1], o[2], o[3]);
            }
          }
        }
        // ---- q (columns 0..63): pulled into registers, then the accumulator is free for the next tile's MMAs ----
        uint32_t q0[32], q1[32];
        umma::ld_32x32b_x32(t_row, q0);
        umma::ld_32x32b_x32(t_row + 32u, q1);
        umma::ld_wait32(q0);
        umma::ld_wait32(q1);
        umma::fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tmem_empty);
        acc_phase ^= 1u;
        // softmax over the 32 channels of a head, scaled; this thread's two heads
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          float f[32];
          float m = -INFINITY;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 a = lds4(tq_s + (uint32_t)(hh * 32 + 4 * j4) * 4u);
            const float ta[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int j = 4 * j4 + i;
              f[j] = fmaf(__uint_as_float(hh == 0 ? q0[j] : q1[j]), rl2, ta[i]);
              m = fmaxf(m, f[j]);
            }
          }
          float sum = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(f[j]) : "f"(f[j] - m));
            sum += f[j];
          }
          const float inv = P.scale / sum;
          if (valid) {
            act_t* dst = P.qout + ((size_t)n * P.npix + p0 + row) * AQ_HID + (hp * 2 + hh) * AQ_DH;
#pragma unroll
            for (int v = 0; v < 2; ++v) {
              uint4 a, b;
              a.x = pack_q(f[16 * v + 0] * inv, f[16 * v + 1] * inv);   a.y = pack_q(f[16 * v + 2] * inv, f[16 * v + 3] * inv);
              a.z = pack_q(f[16 * v + 4] * inv, f[16 * v + 5] * inv);   a.w = pack_q(f[16 * v + 6] * inv, f[16 * v + 7] * inv);
              b.x = pack_q(f[16 * v + 8] * inv, f[16 * v + 9] * inv);   b.y = pack_q(f[16 * v + 10] * inv, f[16 * v + 11] * inv);
              b.z = pack_q(f[16 * v + 12] * inv, f[16 * v + 13] * inv); b.w = pack_q(f[16 * v + 14] * inv, f[16 * v + 15] * inv);
              stg_256(dst + 16 * v, a, b);
            }
          }
        }
        umma::named_bar_sync(2, 128);                            // P and V of this tile are staged
        if (rescale && etid < 2 * AQ_DH) s_dl[etid] = 0.f;       // (every read of this tile's step is behind that barrier)

        // ---- context: S[d][e] += sum_pix P[pix][d] V[pix][e] (and Z[d] through a column of ones), head hl of the pair, d rows 16*mt.. ----
        {
          const uint32_t ones = ((lane >> 2) == 0) ? 0x3F803F80u : 0u;       // B fragment of the ones column: n = 0 for every k
          const uint32_t pa = smem_u32(s_p) + (uint32_t)((lr + ((lmat >> 1) & 1) * 8) * AQ_PITCH + (hl * 32 + mt * 16 + (lmat & 1) * 8) * 2);
          const uint32_t vb = smem_u32(s_v) + (uint32_t)((lr + (lmat & 1) * 8) * AQ_PITCH + (hl * 32 + (lmat >> 1) * 8) * 2);
#pragma unroll
          for (int ks = 0; ks < AQ_TILE / 16; ++ks) {
            uint32_t a[4], b01[4], b23[4];
            ldsm_x4_trans(a, pa + (uint32_t)(ks * 16 * AQ_PITCH));
            ldsm_x4_trans(b01, vb + (uint32_t)(ks * 16 * AQ_PITCH));
            ldsm_x4_trans(b23, vb + (uint32_t)(ks * 16 * AQ_PITCH + 32));
            mma_bf16(c[0], a, b01[0], b01[1]);
            mma_bf16(c[1], a, b01[2], b01[3]);
            mma_bf16(c[2], a, b23[0], b23[1]);
            mma_bf16(c[3], a, b23[2], b23[3]);
            mma_bf16(cz, a, ones, ones);
          }
        }
        umma::named_bar_sync(2, 128);                            // every warp is past its context MMAs: the staging rows are free
      }
      // ---- one partial per (sample, head, chunk): S rows d = 16 mt + {g, g + 8}, Z from the ones column,
      //      m[d] in natural-log units as attn_reduce_kernel expects ----
      {
        float* po = P.part + (((size_t)n * AQ_HEADS + hp * 2 + hl) * P.chunks + chunk) * AQ_PART;
        const int g = lane >> 2, q = lane & 3;
        const int d = mt * 16 + g;
#pragma unroll
        for (int nt8 = 0; nt8 < 4; ++nt8) {
          *reinterpret_cast<float2*>(po + d * AQ_DH + nt8 * 8 + q * 2) = make_float2(c[nt8][0], c[nt8][1]);
          *reinterpret_cast<float2*>(po + (d + 8) * AQ_DH + nt8 * 8 + q * 2) = make_float2(c[nt8][2], c[nt8][3]);
        }
        if (q == 0) { po[AQ_DH * AQ_DH + d] = cz[0]; po[AQ_DH * AQ_DH + d + 8] = cz[2]; }
        if (lane < 16) po[AQ_DH * AQ_DH + AQ_DH + mt * 16 + lane] = s_m[hl * AQ_DH + mt * 16 + lane] * kLn2;
      }
    }
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 2) { umma::fence_after(); umma::tmem_dealloc(tmem_base, 256); }
}

}  // namespace ds

using namespace ds;

extern "C" {

/* Fused PreNorm + to_qkv + q soft-max + partial linear-attention context of the U-Net attention (hidden = 4 heads x 32).
   d_x act16 NHWC [x_batch_mod or N][npix][C]; d_weight act16 [384][C] (rows q | k | v, GroupNorm gamma folded in);
   d_e1 / d_e2 fp32 [384] (the fold's tables, e1 nullable), d_stats_in the statistics buffer of x (nullable: no norm);
   d_sbias fp32 [N][sbias_stride] (label_query | label_key | 0; nullable).  Outputs: d_q_out act16 [N][npix][128] = softmax_d(q) * scale,
   d_part = chunk partials in the layout of ds_attn_ctx_partial (ds_attn_part_floats floats; ds_attn_finalize merges them). */
int ds_attn_qkv_ctx(const void* d_x, int C, int x_batch_mod, const void* d_stats_in, int stats_in_slots, const void* d_weight,
                    const float* d_e1, const float* d_e2, const float* d_sbias, long long sbias_stride, void* d_q_out, float* d_part,
                    int N, int heads, long long npix, float scale, void* stream) {
  DS_REQUIRE(d_x && d_weight && d_e2 && d_q_out && d_part && N > 0 && npix > 0, "ds_attn_qkv_ctx: bad arguments");
  DS_REQUIRE(heads == AQ_HEADS, "ds_attn_qkv_ctx: heads=%d (only the U-Net's 4 heads x 32 are built)", heads);
  DS_REQUIRE(C > 0 && C % AQ_BK == 0, "ds_attn_qkv_ctx: C=%d must be a multiple of %d", C, AQ_BK);
  DS_REQUIRE(!d_stats_in || d_e1, "ds_attn_qkv_ctx: stats_in needs e1");
  DS_REQUIRE(npix < (1ll << 30) && (long long)N * ds_attn_chunks(npix) < (1ll << 29), "ds_attn_qkv_ctx: problem too large");
  EncodeTiledFn encode = get_encode_fn();
  DS_REQUIRE(encode != nullptr, "ds_attn_qkv_ctx: cuTensorMapEncodeTiled entry point not available");
  const CUtensorMapDataType dt = kOperandIsFp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap map_a, map_b;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)npix, (cuuint64_t)(x_batch_mod > 0 ? x_batch_mod : N)};
    const cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)npix * C * 2};
    const cuuint32_t box[3] = {AQ_BK, AQ_TILE, 1}, estr[3] = {1, 1, 1};
    const CUresult r = encode(&map_a, dt, 3, const_cast<void*>(d_x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DS_REQUIRE(r == CUDA_SUCCESS, "ds_attn_qkv_ctx: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
  }
  {
    const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)AQ_NOUT, 1};
    const cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)AQ_NOUT * C * 2};
    const cuuint32_t box[3] = {AQ_BK, 2 * AQ_DH, 1}, estr[3] = {1, 1, 1};
    const CUresult r = encode(&map_b, dt, 3, const_cast<void*>(d_weight), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DS_REQUIRE(r == CUDA_SUCCESS, "ds_attn_qkv_ctx: cuTensorMapEncodeTiled(weight) failed with %d", (int)r);
  }
  AttnQkvDev P;
  memset(&P, 0, sizeof(P));
  P.N = N; P.npix = (int)npix; P.C = C; P.num_kb = C / AQ_BK; P.x_batch_mod = x_batch_mod;
  P.chunks = ds_attn_chunks(npix);
  P.items = N * P.chunks * 2;      // x 2 head pairs
  P.stats_in = reinterpret_cast<const float2*>(d_stats_in); P.stats_in_slots = stats_in_slots;
  P.e1 = d_e1; P.e2 = d_e2; P.sbias = d_sbias; P.sbias_stride = sbias_stride;
  P.qout = reinterpret_cast<act_t*>(d_q_out); P.part = d_part; P.scale = scale;
  DS_CHECK_CUDA(cudaFuncSetAttribute(attn_qkv_ctx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AQ_SMEM));
  const int grid = P.items < 2 * num_sms() ? P.items : 2 * num_sms();      // two resident CTAs per SM
  DS_CHECK_CUDA(launch_pdl(attn_qkv_ctx_kernel, dim3(grid), dim3(AQ_THREADS), (size_t)(AQ_SMEM), (cudaStream_t)stream, map_a, map_b, P));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
