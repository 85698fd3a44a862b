// Depthwise 7x7 convolution (ConvNextBlock.ds_conv, model/diffusion_components.py:118,131) fused with the
// per-sample time-embedding bias (:133-136) and the (sum, sumsq) partials of the GroupNorm(1,C) that
// follows (:121), and the 7x7 stem convolution (init_conv, model/diffusion.py:82).
#include "common.cuh"
#include "../../include/diffusynth_b200.h"
#include "tma.cuh"
#include <cstdlib>

namespace ds {

// ---------------------------------------------------------------------------------------------
// dwconv7: 16-bit NHWC in (one or two channel-concatenated sources), 16-bit NHWC out.
// block = 256 threads = 16 channel pairs x 16 pixel-threads; tile = (8*R) rows x 16 cols x 32 channels, R = 1 or 2.
// (A warp-level tensor-core formulation -- mma.sync m16n8k16 with block-diagonal weight fragments, 1/8 of the lanes
// useful -- was measured on B200 at 9.6 ms per U-Net evaluation against 6.4 ms for the R=1 kernel: legacy HMMA is too slow
// on sm_100a to pay for the 8x redundancy.  See profiles/r01_notes.md.)
// The (8R+6) x (16+6) halo tile is staged in shared memory as fp32 (row pitch padded to 23 pixels); each thread slides a
// 7-wide window over R rows x 8 output columns with packed FFMA2.  With R = 1 the kernel is bound by shared-memory
// bandwidth (21 LDS.64 per 56 FFMA2); with R = 2 every staged input row feeds two output rows and each weight row is
// loaded once, which brings the LDS traffic under the FMA-pipe time.
// ---------------------------------------------------------------------------------------------
static constexpr int DW_TW = 16, DW_CB = 32;
static constexpr int DW_HW = DW_TW + 6, DW_PITCH = 23;

template <int R>
__global__ void __launch_bounds__(256, R == 1 ? 4 : 3)
dwconv7_kernel(const act_t* __restrict__ src0, const act_t* __restrict__ src1, int C0, int C1, int src_batch_mod,
               const float* __restrict__ weight,   // [49][C] (tap-major)
               const float* __restrict__ tbias, long long tbias_stride,   // [N or 1][>=C]: conv bias + time projection
               act_t* __restrict__ out, float2* __restrict__ stats, float stats_inv_count, float eps, int H, int W, int tiles_w, int tiles) {
  pdl_enter();
  constexpr int TH = 8 * R, HH = TH + 6;
  extern __shared__ __align__(16) float2 dw_smem[];
  float2* s_in = dw_smem;                                   // [HH][DW_PITCH][16] fp32 channel pairs (converted once at staging)
  float2* s_w = dw_smem + HH * DW_PITCH * (DW_CB / 2);      // [49][16]
  __shared__ float s_red[16];
  const int C = C0 + C1;
  const int tile = blockIdx.x, cblk = blockIdx.y, n = blockIdx.z;
  const int h0 = (tile / tiles_w) * TH, w0 = (tile % tiles_w) * DW_TW;
  const int c0 = cblk * DW_CB;
  const int nsrc = (src_batch_mod > 0 && c0 < C0) ? n % src_batch_mod : n;      // the batch modulus applies to source 0 only
  const act_t* src;
  int Cs, cs0;
  if (c0 < C0) { src = src0; Cs = C0; cs0 = c0; } else { src = src1; Cs = C1; cs0 = c0 - C0; }
  src += (size_t)nsrc * H * W * Cs;

  // stage weights: s_w[tap][cp] = (w[tap][c0+2cp], w[tap][c0+2cp+1])
  for (int i = threadIdx.x; i < 49 * (DW_CB / 2); i += 256) {
    const int tap = i / (DW_CB / 2), cp = i % (DW_CB / 2);
    s_w[i] = make_float2(__ldg(weight + (size_t)tap * C + c0 + 2 * cp), __ldg(weight + (size_t)tap * C + c0 + 2 * cp + 1));
  }
  // stage the halo tile: 16-byte pieces (8 channels) per thread, converted to fp32 once; 4 pieces per pixel
  for (int i = threadIdx.x; i < HH * DW_HW * 4; i += 256) {
    const int piece = i & 3, pix = i >> 2;
    const int r = pix / DW_HW, cc = pix - r * DW_HW;
    const int y = h0 + r - 3, x = w0 + cc - 3;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (y >= 0 && y < H && x >= 0 && x < W)
      v = __ldg(reinterpret_cast<const uint4*>(src + ((size_t)y * W + x) * Cs + cs0 + piece * 8));
    float4* dst = reinterpret_cast<float4*>(&s_in[(r * DW_PITCH + cc) * (DW_CB / 2) + piece * 4]);
    const float2 a = cvt16x2(v.x), b = cvt16x2(v.y), c = cvt16x2(v.z), d = cvt16x2(v.w);
    dst[0] = make_float4(a.x, a.y, b.x, b.y);
    dst[1] = make_float4(c.x, c.y, d.x, d.y);
  }
  __syncthreads();

  const int cp = threadIdx.x & 15, pt = threadIdx.x >> 4;
  const int row0 = (pt & 7) * R, col0 = (pt >> 3) * 8;
  float2 acc[R][8];    // (channel 2cp, channel 2cp+1) of R rows x 8 consecutive output columns: packed FFMA2 lanes
#pragma unroll
  for (int i = 0; i < R; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = make_float2(0.f, 0.f);
  float2 wbuf[R][7];   // weight rows ky = r, r-1, .., r-R+1 (slot ky % R)
#pragma unroll
  for (int r = 0; r < R + 6; ++r) {
    if (r < 7) {
#pragma unroll
      for (int kx = 0; kx < 7; ++kx) wbuf[r % R][kx] = s_w[(r * 7 + kx) * (DW_CB / 2) + cp];
    }
    const float2* rowp = &s_in[((row0 + r) * DW_PITCH + col0) * (DW_CB / 2) + cp];
#pragma unroll
    for (int j = 0; j < 14; ++j) {
      const float2 in = rowp[j * (DW_CB / 2)];
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const int ky = r - i;
        if (ky >= 0 && ky < 7) {
#pragma unroll
          for (int kx = 0; kx < 7; ++kx) {
            const int ow = j - kx;
            if (ow >= 0 && ow < 8) ffma2(acc[i][ow], in, wbuf[ky % R][kx]);
          }
        }
      }
    }
  }
  const int c = c0 + 2 * cp;
  const float* tb = tbias + (size_t)(tbias_stride ? n : 0) * tbias_stride;
  const float b0 = __ldg(tb + c), b1 = __ldg(tb + c + 1);
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int y = h0 + row0 + i;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int x = w0 + col0 + j;
      if (y < H && x < W) {
        const float v0 = acc[i][j].x + b0, v1 = acc[i][j].y + b1;
        s += v0 + v1;
        q = fmaf(v0, v0, fmaf(v1, v1, q));
        *reinterpret_cast<uint32_t*>(out + (((size_t)n * H + y) * W + x) * C + c) = pack16(v0, v1);
      }
    }
  }
  if (stats != nullptr) {
    s = warp_sum(s);
    q = warp_sum(q);
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_red[warp] = s; s_red[8 + warp] = q; }
    __syncthreads();
    if (threadIdx.x < 32) {
      float ts = 0.f, tq = 0.f;
      if (threadIdx.x == 0)
        for (int i = 0; i < 8; ++i) { ts += s_red[i]; tq += s_red[8 + i]; }
      const int slots = tiles * gridDim.y;
      stats_publish(stats_sample(stats, slots, n), slots, cblk * tiles + tile, ts, tq, stats_inv_count, eps, threadIdx.x);
    }
  }
}

// halo tile of the tensor-core kernel below: one cp.async.bulk.tensor box of 22 x 22 pixels x 32 channels (out-of-range rows and
// columns zero-filled by the TMA unit = the conv padding), two stages
static constexpr int DT_HALO = 22, DT_STAGES = 2;
static constexpr int DT_TILE_BYTES = DT_HALO * DT_HALO * DW_CB * 2;     // 30976, a multiple of 128

// ---------------------------------------------------------------------------------------------
// dwconv7 on the warp-level tensor cores (mma.sync.m16n8k16, fp32 accumulate), Toeplitz formulation.
// A depthwise convolution has no channel contraction, so the block-diagonal GEMM (M = pixels, K = taps x channels) wastes 7/8
// of every MMA (measured: slower than FFMA2, see above).  Here the contraction runs over the INPUT COLUMN instead: for one
// channel and one kernel row dy,   out[y, x] += sum_k In[y + dy, k] * T_dy[k, x],   T_dy[k, x] = w[dy][k - x] (0 <= k - x <= 6),
// i.e. a [16 rows x 16 input columns] x [16 x 8] product per 16 x 8 outputs: 7 of the 16 k of every row of T are non-zero for
// every output column (44 % of the MMA is useful work), 14 MMAs per channel and 16 x 16 output tile instead of 784 FFMA2 lanes.
// The operands of such an MMA are x-contiguous for a fixed channel, the tensors are channels-last: each TMA-staged halo tile
// [22 y][22 x][32 c] is first transposed into per-channel planes [c][22 y][24 x] with ldmatrix.trans (an 8 pixels x 8 channels
// block per matrix), the fp32 results go back through per-channel planes [c][16 y][16 x] and a second ldmatrix.trans that
// yields channel pairs per pixel for the channels-last stores.  A warp owns 4 of the block's 32 channels and keeps their
// 7 x 2 Toeplitz B fragments in registers for the whole (persistent) kernel.  Plane pitches (1072 / 528 bytes) make every
// ldmatrix and every 32-bit plane store conflict-free.  The output planes alias the raw stage that was just transposed.
// ---------------------------------------------------------------------------------------------
static constexpr int DM_PLANE = 22 * 48 + 16;      // bytes per input plane: 22 rows of 24 halves, padded
static constexpr int DM_OPLANE = 16 * 32 + 16;     // bytes per output plane: 16 rows of 16 halves, padded
static constexpr int DM_SMEM_BYTES = DT_STAGES * DT_TILE_BYTES + DW_CB * DM_PLANE + DW_CB * DM_OPLANE + 64 + DT_STAGES * 8 + 128;

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
#ifdef DS_OPERANDS_BF16
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
#else
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
#endif
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack16_sat(float lo, float hi) {
#ifdef DS_OPERANDS_BF16
  return pack16(lo, hi);
#else
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
#endif
}
// address of 16-byte chunk `chunk` of 64-byte row `row` of a TMA SWIZZLE_64B box at `base`: address bits [4:5] ^= bits [7:8]
__device__ __forceinline__ uint32_t swz64(uint32_t base, int row, int chunk) {
  const uint32_t a = base + (uint32_t)(row * 64 + chunk * 16);
  return a ^ (((a >> 7) & 3u) << 4);
}

__global__ void __launch_bounds__(256, 2)
dwconv7_mma_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1, int C0, int C1, int src_batch_mod,
                   const float* __restrict__ weight, const float* __restrict__ tbias, long long tbias_stride,
                   act_t* __restrict__ out, float2* __restrict__ stats, float stats_inv_count, float eps, int H, int W, int tiles_w,
                   int tiles, int N, int dbg_arg) {
  // phase switches for timing experiments (1 skip the MMAs, 2 the output stores, 4 the statistics, 8 the transposes): compiled in
  // only with -DDS_CONV_DEBUG (DS_DW_DBG=<mask>), a constant 0 otherwise
#ifdef DS_CONV_DEBUG
  const int dbg = dbg_arg;
#else
  constexpr int dbg = 0;
  (void)dbg_arg;
#endif
  extern __shared__ uint8_t dm_smem_raw[];
  uint8_t* smem = dm_smem_raw + ((128u - (smem_u32(dm_smem_raw) & 127u)) & 127u);
  const uint32_t s_raw = smem_u32(smem);                                      // [stage][22 y][22 x][32 c] halves, 64B-swizzled by the TMA unit
  const uint32_t s_plane = s_raw + DT_STAGES * DT_TILE_BYTES;                 // [32 c][DM_PLANE]
  const uint32_t s_oplane = s_plane + DW_CB * DM_PLANE;                       // [32 c][DM_OPLANE]
  const uint32_t s_zero = s_oplane + DW_CB * DM_OPLANE;                       // 64 zero bytes
  uint8_t* tail = smem + DT_STAGES * DT_TILE_BYTES + DW_CB * DM_PLANE + DW_CB * DM_OPLANE;
  uint64_t* full = reinterpret_cast<uint64_t*>(tail + 64);
  __shared__ float s_red[2][16];
  const int C = C0 + C1;
  const int cblk = blockIdx.y, c0 = cblk * DW_CB;
  const CUtensorMap* map = c0 < C0 ? &map0 : &map1;
  const int cs0 = c0 < C0 ? c0 : c0 - C0;
  const int total = N * tiles;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;

  if (threadIdx.x == 0) {
    prefetch_tmap(map);
    for (int s = 0; s < DT_STAGES; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 16) reinterpret_cast<uint32_t*>(tail)[threadIdx.x] = 0u;

  // Toeplitz B fragments of this warp's 4 channels.  b0 holds T[k = 2q (+1)][n = g], b1 holds T[k = 2q + 8 (+1)][n = g] with
  // T[k][n] = w[dy][k - n] for 0 <= k - n <= 6: b0 is non-zero only for g <= 2q + 1 and b1 only for g >= 2q + 2, so one register
  // per (channel, kernel row) and two lane masks carry both.
  const uint32_t m0 = g <= 2 * q + 1 ? 0xffffffffu : 0u, m1 = ~m0;
  uint32_t bfr[4][7];
#pragma unroll
  for (int ci = 0; ci < 4; ++ci) {
    const int c = c0 + 4 * warp + ci;
#pragma unroll
    for (int dy = 0; dy < 7; ++dy) {
      const int d0 = 2 * q - g + (m0 ? 0 : 8), d1 = d0 + 1;
      const float w0 = (d0 >= 0 && d0 < 7) ? __ldg(weight + (size_t)(dy * 7 + d0) * C + c) : 0.f;
      const float w1 = (d1 >= 0 && d1 < 7) ? __ldg(weight + (size_t)(dy * 7 + d1) * C + c) : 0.f;
      bfr[ci][dy] = pack16(w0, w1);
    }
  }
  pdl_launch_dependents();
  pdl_wait();
  __syncthreads();

  auto issue = [&](int item, int stage) {
    const int n = item / tiles, t = item - n * tiles;
    const int th = t / tiles_w, tw = t - th * tiles_w;
    const int nsrc = (src_batch_mod > 0 && c0 < C0) ? n % src_batch_mod : n;
    mbar_expect_tx(&full[stage], DT_TILE_BYTES);
    tma_load_4d(smem + stage * DT_TILE_BYTES, map, &full[stage], cs0, tw * DW_TW - 3, th * 16 - 3, nsrc);
  };
  // each block walks a contiguous run of (sample, tile) items: neighbouring halos stay in L2 and the statistics of a sample
  // are published once per run instead of once per tile
  const int per_block = (total + (int)gridDim.x - 1) / (int)gridDim.x;
  const int item0 = blockIdx.x * per_block, item1 = min(item0 + per_block, total);
  if (threadIdx.x == 0) {
    if (item0 < item1) issue(item0, 0);
    if (item0 + 1 < item1) issue(item0 + 1, 1);
  }
  int run_len = 0;      // warp 0: tiles of the current sample whose statistics slots are written but not yet announced

  const int a_row = (lane & 7) + ((lane >> 3) & 1) * 8, a_chunk = lane >> 4;
  const uint32_t pl2 = s_plane + (uint32_t)(a_row * 48 + 32);      // ldmatrix.x2: lanes 0-15 address rows 0-15 of columns 16-23
  const int t_i = lane & 7, t_j = lane >> 3;                 // transposes: lane supplies row t_i of matrix t_j
  int it = 0;
  for (int item = item0; item < item1; ++item, ++it) {
    const int stage = it & 1;
    const int n = item / tiles, t = item - n * tiles;
    const int h0 = (t / tiles_w) * 16, w0 = (t % tiles_w) * DW_TW;
    const float* tb = tbias + (size_t)(tbias_stride ? n : 0) * tbias_stride;
    // this warp's four bias values: requested before the wait for the tile so that the global-load latency hides behind the TMA wait and
    // the transposes (issued at their first use, between two shared-memory phases, they showed up as long-scoreboard stalls on the
    // accumulator initialisation)
    float bias4[4];
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) bias4[ci] = __ldg(tb + c0 + 4 * warp + ci);
    mbar_wait(&full[stage], (uint32_t)(it >> 1) & 1u);
    const uint32_t raw = s_raw + stage * DT_TILE_BYTES;

    // ---- channels-last halo tile -> per-channel planes.  Warp w takes rows w, w + 8, w + 16; per row three 8-pixel groups; one
    // ldmatrix.x4.trans per group: matrix j = channel chunk j, its 8 rows = the 8 pixels; afterwards lane (g, q) holds pixels
    // (2q, 2q + 1) of channel 8j + g.
    for (int y = warp; y < ((dbg & 8) ? 0 : DT_HALO); y += 8) {
      const uint32_t dst = s_plane + (uint32_t)(g * DM_PLANE + y * 48 + q * 4);
#pragma unroll
      for (int xg = 0; xg < 3; ++xg) {
        const int x = 8 * xg + t_i;
        const uint32_t addr = (xg < 2 || x < DT_HALO) ? swz64(raw, y * DT_HALO + x, t_j) : s_zero;
        uint32_t r[4];
        ldsm_x4_t(r, addr);
#pragma unroll
        for (int j = 0; j < 4; ++j) sts32(dst + (uint32_t)(8 * j * DM_PLANE + xg * 16), r[j]);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();          // planes complete; this raw stage is free again; everyone is done with the previous output planes
    if (threadIdx.x == 0 && item + 2 < item1) issue(item + 2, stage);

    // ---- 4 channels per warp, two at a time: 7 kernel rows x 2 column halves of m16n8k16 each
    const bool full_tile = h0 + 16 <= H && w0 + DW_TW <= W;
    float s = 0.f, sq = 0.f;
#pragma unroll
    for (int cp = 0; cp < 2; ++cp) {
      float d[2][2][4];
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const float bias = bias4[2 * cp + cc];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int k = 0; k < 4; ++k) d[cc][h][k] = bias;
      }
#pragma unroll
      for (int dy = 0; dy < 7; ++dy) {
        if (dbg & 1) break;
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int ci = 2 * cp + cc;
          const uint32_t pl = s_plane + (uint32_t)((4 * warp + ci) * DM_PLANE + (a_row + dy) * 48 + a_chunk * 16);
          uint32_t a[4], e2[2];
          ldsm_x4(a, pl);            // rows 0-7 / 8-15 of input columns 0-7 and 8-15
          ldsm_x2(e2, pl2 + (uint32_t)((4 * warp + ci) * DM_PLANE + dy * 48));      // the same rows of input columns 16-23
          const uint32_t e[4] = {a[2], a[3], e2[0], e2[1]};      // (shared memory is the busiest unit: 6 matrices per kernel row, not 8)
          const uint32_t b0 = bfr[ci][dy] & m0, b1 = bfr[ci][dy] & m1;
          mma16816(d[cc][0], a, b0, b1);      // output columns 0-7
          mma16816(d[cc][1], e, b0, b1);      // output columns 8-15
        }
      }
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const uint32_t op = s_oplane + (uint32_t)((4 * warp + 2 * cp + cc) * DM_OPLANE + g * 32 + q * 4);
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const float v0 = d[cc][h][2 * rr], v1 = d[cc][h][2 * rr + 1];
            if (full_tile) {
              s += v0 + v1;
              sq = fmaf(v0, v0, fmaf(v1, v1, sq));
            } else if (h0 + g + 8 * rr < H) {
              const int x = w0 + 8 * h + 2 * q;
              if (x < W) { s += v0; sq = fmaf(v0, v0, sq); }
              if (x + 1 < W) { s += v1; sq = fmaf(v1, v1, sq); }
            }
            sts32(op + (uint32_t)(rr * 8 * 32 + h * 16), pack16_sat(v0, v1));
          }
      }
    }
    float* red = s_red[it & 1];
    if (stats != nullptr) {
      s = warp_sum(s);
      sq = warp_sum(sq);
      if (lane == 0) { red[warp] = s; red[8 + warp] = sq; }
    }
    __syncthreads();          // output planes complete (and the per-warp partials visible); the input planes are free again

    // ---- planes -> channels-last: matrix j = channels 8j..8j+7 of one (row, 8-pixel group); .trans gives channel pairs per pixel
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int y = 2 * warp + (u >> 1), xc = u & 1;
      uint32_t r[4];
      ldsm_x4_t(r, s_oplane + (uint32_t)(lane * DM_OPLANE + y * 32 + xc * 16));      // lane = 8j + i: channel row i of matrix j
      const int yy = h0 + y, xx = w0 + 8 * xc + g;
      if (yy < H && xx < W && !(dbg & 2)) {
        uint32_t* o = reinterpret_cast<uint32_t*>(out + (((size_t)n * H + yy) * W + xx) * C + c0) + q;
#pragma unroll
        for (int j = 0; j < 4; ++j) o[4 * j] = r[j];
      }
    }
    if (stats != nullptr && threadIdx.x < 32 && !(dbg & 4)) {
      const int slots = tiles * gridDim.y;
      float2* sb = stats_sample(stats, slots, n);
      if (threadIdx.x == 0) {
        float ts = 0.f, tq = 0.f;
        for (int i = 0; i < 8; ++i) { ts += red[i]; tq += red[8 + i]; }
        sb[2 + cblk * tiles + t] = make_float2(ts, tq);       // this tile's slot: a plain store, announced with the run
      }
      ++run_len;
      if (t == tiles - 1 || item + 1 == item1) {      // last tile of this sample in the run
        stats_arrive_run(sb, slots, run_len, stats_inv_count, eps, threadIdx.x);
        run_len = 0;
      }
    }
  }
}

static inline int dw_rows_per_thread(int H) { return H >= 16 ? 2 : 1; }      // 16-row tiles (tensor-core kernel) or 8-row tiles
static inline size_t dw_smem_bytes(int R) { return (size_t)((8 * R + 6) * DW_PITCH + 49) * (DW_CB / 2) * sizeof(float2); }

// ---------------------------------------------------------------------------------------------
// Stem as a GEMM: im2col of the 7x7xCin (Cin <= 4) patches into a 16-bit [N, H, W, 224] matrix (k = ky*32 + kx*4 + ci,
// the 8th pixel slot of every ky row is zero) so that init_conv runs as a 1x1 ds_conv_gemm with K = 224 on the tensor cores.
// One thread per (pixel, ky): 64 contiguous output bytes.
// ---------------------------------------------------------------------------------------------
__global__ void stem_im2col_kernel(const float* __restrict__ x, act_t* __restrict__ col, int Cin, int H, int W, long long total /* N*H*W*7 */) {
  pdl_enter();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int xx = (int)(i % W);
    long long r = i / W;
    const int ky = (int)(r % 7); r /= 7;
    const int y = (int)(r % H);
    const long long n = r / H;
    const int sy = y + ky - 3;
    uint32_t packed[16];
#pragma unroll
    for (int kx = 0; kx < 8; ++kx) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      const int sx = xx + kx - 3;
      if (kx < 7 && sy >= 0 && sy < H && sx >= 0 && sx < W) {
#pragma unroll
        for (int ci = 0; ci < 4; ++ci)
          if (ci < Cin) v[ci] = __ldg(x + ((n * Cin + ci) * H + sy) * W + sx);
      }
      packed[2 * kx] = pack16(v[0], v[1]);
      packed[2 * kx + 1] = pack16(v[2], v[3]);
    }
    act_t* dst = col + ((n * H + y) * W + xx) * 224 + ky * 32;       // 64 contiguous bytes: two full 32-byte sectors
#pragma unroll
    for (int q = 0; q < 2; ++q)
      stg_256(dst + 16 * q, make_uint4(packed[8 * q], packed[8 * q + 1], packed[8 * q + 2], packed[8 * q + 3]),
              make_uint4(packed[8 * q + 4], packed[8 * q + 5], packed[8 * q + 6], packed[8 * q + 7]));
  }
}

}  // namespace ds

using namespace ds;

extern "C" {

/* Depthwise 7x7 + time bias + GroupNorm partials.  d_weight fp32 [49][C0+C1] (tap-major);
   d_tbias fp32 [N][tbias_stride] (or one row when tbias_stride == 0) holding ds_conv.bias + mlp(time_emb).
   d_stats (nullable): statistics buffer float2 [N][2 + ds_dwconv7_stats_slots(...)], zero-initialised once (see ds_conv_gemm). */
int ds_dwconv7(const void* d_src0, const void* d_src1, int C0, int C1, int src_batch_mod, const float* d_weight, const float* d_tbias,
               long long tbias_stride, void* d_out, void* d_stats, float eps, int N, int H, int W, void* stream) {
  DS_REQUIRE(d_src0 && d_weight && d_tbias && d_out && N > 0 && H > 0 && W > 0, "ds_dwconv7: bad arguments");
  DS_REQUIRE(C0 > 0 && C0 % DW_CB == 0 && C1 >= 0 && C1 % DW_CB == 0 && (C1 == 0 || d_src1), "ds_dwconv7: C0=%d C1=%d must be multiples of 32", C0, C1);
  const int R = dw_rows_per_thread(H);
  const int tiles_w = (W + DW_TW - 1) / DW_TW, tiles_h = (H + 8 * R - 1) / (8 * R);
  const int tiles = tiles_w * tiles_h;
  const int cblks = (C0 + C1) / DW_CB;
  DS_REQUIRE(N <= 65535 && cblks <= 65535, "ds_dwconv7: grid too large");
  const float inv_count = 1.0f / ((float)H * (float)W * (float)(C0 + C1));
  if (R == 1) {
    // maps shorter than 16 rows (the deepest levels of narrow / low configurations): direct FFMA2 kernel on 8-row tiles
    DS_CHECK_CUDA(cudaFuncSetAttribute(dwconv7_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dw_smem_bytes(1)));
    DS_CHECK_CUDA(launch_pdl((dwconv7_kernel<1>), dim3(tiles, cblks, N), dim3(256), dw_smem_bytes(1), (cudaStream_t)stream,
        (const act_t*)d_src0, (const act_t*)d_src1, C0, C1, src_batch_mod, d_weight, d_tbias, tbias_stride,
        (act_t*)d_out, (float2*)d_stats, inv_count, eps, H, W, tiles_w, tiles));
    return DS_OK;
  }
  EncodeTiledFn encode = get_encode_fn();
  DS_REQUIRE(encode != nullptr, "ds_dwconv7: cuTensorMapEncodeTiled entry point not available");
  CUtensorMap maps[2];      // per call: host threads may launch concurrently
  for (int sidx = 0; sidx < 2; ++sidx) {
    const int nsamp = (sidx == 0 && src_batch_mod > 0) ? src_batch_mod : N;
    const int Cs = sidx == 0 ? C0 : C1;
    const void* base = sidx == 0 ? d_src0 : d_src1;
    if (Cs == 0) { maps[1] = maps[0]; break; }
    const cuuint64_t dims[4] = {(cuuint64_t)Cs, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)nsamp};
    const cuuint64_t strides[3] = {(cuuint64_t)Cs * 2, (cuuint64_t)W * Cs * 2, (cuuint64_t)H * W * Cs * 2};
    const cuuint32_t box[4] = {(cuuint32_t)DW_CB, (cuuint32_t)DT_HALO, (cuuint32_t)DT_HALO, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = encode(&maps[sidx], kOperandIsFp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                              4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DS_REQUIRE(r == CUDA_SUCCESS, "ds_dwconv7: cuTensorMapEncodeTiled failed with %d (C=%d W=%d H=%d)", (int)r, Cs, W, H);
  }
  const long long work = (long long)N * tiles;
  int gm = 2 * num_sms() / cblks;      // never more blocks than resident slots (2 per SM): a straggler wave would cost a whole pass
  if (gm > work) gm = (int)work;
  if (gm < 1) gm = 1;
#ifdef DS_CONV_DEBUG
  static const int dw_dbg = [] { const char* e = getenv("DS_DW_DBG"); return e ? atoi(e) : 0; }();      // phase switches (tools_dev/ab_dwconv.py)
#else
  const int dw_dbg = 0;
#endif
  DS_CHECK_CUDA(cudaFuncSetAttribute(dwconv7_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DM_SMEM_BYTES));
  DS_CHECK_CUDA(launch_pdl(dwconv7_mma_kernel, dim3(gm, cblks), dim3(256), (size_t)DM_SMEM_BYTES, (cudaStream_t)stream,
      maps[0], maps[1], C0, C1, src_batch_mod, d_weight, d_tbias, tbias_stride, (act_t*)d_out, (float2*)d_stats, inv_count, eps,
      H, W, tiles_w, tiles, N, dw_dbg));
  return DS_OK;
}

int ds_dwconv7_stats_slots(int C, int H, int W) {
  const int R = dw_rows_per_thread(H);
  return ((W + DW_TW - 1) / DW_TW) * ((H + 8 * R - 1) / (8 * R)) * (C / DW_CB);
}

/* im2col for the stem (init_conv as a GEMM): d_x fp32 NCHW [N, Cin<=4, H, W] -> d_col act16 [N, H, W, 224]. */
int ds_stem_im2col(const float* d_x, void* d_col, int N, int Cin, int H, int W, void* stream) {
  DS_REQUIRE(d_x && d_col && N > 0 && Cin > 0 && Cin <= 4 && H > 0 && W > 0, "ds_stem_im2col: bad arguments");
  const long long total = (long long)N * H * W * 7;
  DS_CHECK_CUDA(launch_pdl(stem_im2col_kernel, dim3(grid_for(total, 256, 16)), dim3(256), (size_t)(0), (cudaStream_t)stream, d_x, (act_t*)d_col, Cin, H, W, total));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
