// Batched linear convolution (scipy.signal.fftconvolve along the last axis) by uniformly partitioned FFTs: item k of a ragged
// batch, x_k of N_k samples, is convolved with IR h_{h_index[k]} of M samples.  Both are cut into P = 1024-sample blocks, each
// zero-padded to 2048 and transformed to 1025 bins (the 2048-point real transform of pitch.cu, fft_warp.cuh); a 1024-sample block
// convolved with a 1024-sample partition is 2047 samples long, so nothing aliases.  Output segment s of item k is
//   Y_s = sum over q ascending of X_{s-q} * H_q  (0 <= s - q < nbx_k, 0 <= q < Q),
// inverse-transformed to 2047 samples at s * 1024; output sample j is seg_s[j - 1024 s] + seg_{s-1}[j - 1024 (s-1)], a gather in
// that order.  No float atomics and no per-batch state: an item's result does not depend on the rest of the batch.  Launches:
// forward transforms (signal blocks and IR partitions in one grid), spectral accumulation + inverse, overlap-add gather, and
// the peak scale of pitch.cu when normalising; one metadata copy, no host synchronisation.
#include "common.cuh"
#include "fft_warp.cuh"
#include <climits>
#include <cmath>
#include <vector>
#include "../../include/diffusynth_b200.h"

namespace ds {
namespace {

constexpr int PART = 1024, NFFT = 2048, NC = 1024, NBIN = NFFT / 2 + 1;
constexpr int R = NC / 32;                      // points per lane
constexpr int XS_PITCH = NC + NC / R;           // staging row (fft_warp.cuh), >= NBIN
constexpr int WPB = 8;                          // warps (blocks, segments) per thread block
constexpr int OUT_TILE = 1024;                  // output samples per gather block (one peak partial each)
constexpr int OUT_SPT = OUT_TILE / 256;

// ---- forward transforms: row g of the spectra is block g - foff[u] of source u (u < B: signal u in x, else IR u - B in h),
// samples soff[u] + 1024 t .. + 1023 (zero past slen[u]) zero-padded to 2048; one row per warp. ---------------------------------
__global__ void __launch_bounds__(256)
conv_forward_kernel(const float* __restrict__ x, const float* __restrict__ h, const long long* __restrict__ foff,
                    const long long* __restrict__ soff, const long long* __restrict__ slen, int B, int U, float2* __restrict__ spec,
                    const float2* __restrict__ tw1024, const float2* __restrict__ tw2048) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t cf_smem[];
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(cf_smem);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long g = (long long)blockIdx.x * WPB + w;
  if (g >= __ldg(foff + U)) return;                      // whole warps leave: the transform is warp-local
  const int u = find_item(foff, U, g);
  const long long t0 = (g - __ldg(foff + u)) * PART, L = __ldg(slen + u);
  const float* src = (u < B ? x : h) + __ldg(soff + u);
  float2 v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const long long s0 = t0 + 2 * (lane + 32 * r);
    v[r] = r < R / 2 ? make_float2(s0 < L ? __ldg(src + s0) : 0.f, s0 + 1 < L ? __ldg(src + s0 + 1) : 0.f) : make_float2(0.f, 0.f);
  }
  fft_warp<-1, R>(v, tw1024, lane);
  store_bitrev<R>(xs[w], v, lane);
  __syncwarp();
  rfft2048_unpack<R>(xs[w], spec + g * NBIN, tw2048, lane);
}

// ---- spectral accumulation and inverse: segment g (item k, s = slo[k] + g - goff[k]) sums X_{s-q} H_q over q ascending, lane l
// owning bins l + 32 r (and every lane the Nyquist bin), then irfft -> seg[g][0, 2048) (the last sample is 0 up to rounding).
// Consecutive warps of a block take consecutive segments of one item, so they read the same H_q and overlapping X rows.
__device__ __forceinline__ void cmac(float2& y, float2 a, float2 b) {
  y.x = fmaf(a.x, b.x, fmaf(-a.y, b.y, y.x));
  y.y = fmaf(a.x, b.y, fmaf(a.y, b.x, y.y));
}
__global__ void __launch_bounds__(256)
conv_accumulate_kernel(const float2* __restrict__ spec, float* __restrict__ seg, const long long* __restrict__ foff,
                       const long long* __restrict__ goff, const long long* __restrict__ slo, const long long* __restrict__ hrow,
                       const long long* __restrict__ hq, int B, const float2* __restrict__ tw1024, const float2* __restrict__ tw2048) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t ca_smem[];
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(ca_smem);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long g = (long long)blockIdx.x * WPB + w;
  if (g >= __ldg(goff + B)) return;
  const int k = find_item(goff, B, g);
  const long long s = __ldg(slo + k) + g - __ldg(goff + k), x0 = __ldg(foff + k), nbx = __ldg(foff + k + 1) - x0, Q = __ldg(hq + k);
  const long long qlo = s - (nbx - 1) > 0 ? s - (nbx - 1) : 0, qhi = s < Q - 1 ? s : Q - 1;
  const float2* X = spec + (x0 + s) * NBIN + lane;
  const float2* Hs = spec + __ldg(hrow + k) * NBIN + lane;
  float2 y[R], yn = make_float2(0.f, 0.f);
#pragma unroll
  for (int r = 0; r < R; ++r) y[r] = make_float2(0.f, 0.f);
  for (long long q = qlo; q <= qhi; ++q) {
    const float2* xq = X - q * NBIN;
    const float2* hq_ = Hs + q * NBIN;
#pragma unroll
    for (int r = 0; r < R; ++r) cmac(y[r], __ldg(xq + 32 * r), __ldg(hq_ + 32 * r));
    cmac(yn, __ldg(xq + NC - lane), __ldg(hq_ + NC - lane));
  }
  float2* row = xs[w];
#pragma unroll
  for (int r = 0; r < R; ++r) row[lane + 32 * r] = y[r];
  if (lane == 0) row[NC] = yn;
  __syncwarp();
  float2 v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int b = lane + 32 * r;
    v[r] = irfft2048_pack(row[b], row[NC - b], tw2048, b);
  }
  __syncwarp();
  fft_warp<+1, R>(v, tw1024, lane);
  store_bitrev<R>(row, v, lane);
  __syncwarp();
  float2* out = reinterpret_cast<float2*>(seg + g * NFFT);
  for (int n = lane; n < NC; n += 32) {
    const float2 z = row[pidx<R>(n)];
    out[n] = make_float2(z.x * (1.0f / NFFT), z.y * (1.0f / NFFT));
  }
}

// ---- overlap-add gather and crop: packed output j of item k is full index jf = ostart[k] + j - ooff[k], s = jf / 1024:
// seg_s[jf - 1024 s] + seg_{s-1}[jf - 1024 (s-1)] (a segment outside the item's computed range counts as 0), then
// fl(out[j] + that) when accumulating.  One block per OUT_TILE outputs, each writing its max |out| partial when `peak` is set.
__global__ void __launch_bounds__(256)
conv_output_kernel(const float* __restrict__ seg, float* __restrict__ out, const long long* __restrict__ ooff,
                   const long long* __restrict__ ostart, const long long* __restrict__ goff, const long long* __restrict__ slo, int B,
                   int accumulate, float* __restrict__ peak) {
  pdl_enter();
  __shared__ float red[8];
  const long long total = __ldg(ooff + B);
  float pk = 0.f;
#pragma unroll
  for (int i = 0; i < OUT_SPT; ++i) {
    const long long j = (long long)blockIdx.x * OUT_TILE + threadIdx.x + 256 * i;
    if (j >= total) break;
    const int k = find_item(ooff, B, j);
    const long long jf = __ldg(ostart + k) + j - __ldg(ooff + k), s = jf / PART, r = jf - s * PART;
    const long long lo = __ldg(slo + k), g0 = __ldg(goff + k), n = __ldg(goff + k + 1) - g0;
    const float a = s - lo < n ? __ldg(seg + (g0 + s - lo) * NFFT + r) : 0.f;
    const float b = s - 1 >= lo ? __ldg(seg + (g0 + s - 1 - lo) * NFFT + r + PART) : 0.f;
    float v = a + b;
    if (accumulate) v = out[j] + v;
    out[j] = v;
    pk = fmaxf(pk, fabsf(v));
  }
  if (!peak) return;
  pk = warp_max(pk);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = pk;
  __syncthreads();
  if (threadIdx.x < 32) {
    pk = warp_max(threadIdx.x < 8 ? red[threadIdx.x] : 0.f);
    if (threadIdx.x == 0) peak[blockIdx.x] = pk;
  }
}

// Host plan: the checks, then one int64 metadata array staged at the start of the workspace --
//   foff[B+H+1]  spectrum-row prefix over the B signals then the H IRs (ceil(len / 1024) rows each)
//   soff[B+H]    sample offset of each signal in d_x / IR in d_h;  slen[B+H] their lengths
//   goff[B+1]    segment prefix (item k computes segments slo[k] .. slo[k] + goff[k+1] - goff[k] - 1)
//   slo[B], hrow[B] (first spectrum row of item k's IR), hq[B] (its partition count)
//   ooff[B+1]    output prefix;  ostart[B]
// -- then the spectra (complex64 [rows][1025]), the segments (fp32 [segments][2048]) and, with a peak, one partial per tile.
struct ConvPlan {
  std::vector<long long> meta;
  Workspace ws;
  size_t off_spec = 0, off_seg = 0, off_peak = 0;
  long long n_rows = 0, n_seg = 0, n_out = 0;
  int n_tiles = 0;
  long long *foff = nullptr, *soff = nullptr, *slen = nullptr, *goff = nullptr, *slo = nullptr, *hrow = nullptr, *hq = nullptr,
            *ooff = nullptr, *ostart = nullptr;
};

int plan_conv(const long long* x_lengths, int B, const long long* h_lengths, int H, const long long* h_index, const long long* out_start,
              const long long* out_lengths, float target_peak, const char* who, ConvPlan& p) {
  DS_REQUIRE(x_lengths && h_lengths && h_index && out_start && out_lengths,
             "%s: x_lengths, h_lengths, h_index, out_start and out_lengths must be non-null", who);
  DS_REQUIRE(B > 0 && H > 0, "%s: B = %d and H = %d (both must be > 0)", who, B, H);
  DS_REQUIRE(std::isfinite(target_peak) && target_peak >= 0.f, "%s: target_peak %g (must be finite and >= 0)", who, (double)target_peak);
  for (int i = 0; i < H; ++i) DS_REQUIRE(h_lengths[i] > 0, "%s: impulse response %d has length %lld (must be > 0)", who, i, h_lengths[i]);
  for (int k = 0; k < B; ++k) {
    DS_REQUIRE(x_lengths[k] > 0, "%s: item %d has length %lld (must be > 0)", who, k, x_lengths[k]);
    DS_REQUIRE(h_index[k] >= 0 && h_index[k] < H, "%s: item %d has h_index %lld (must be in [0, %d))", who, k, h_index[k], H);
    const long long full = x_lengths[k] + h_lengths[h_index[k]] - 1;
    DS_REQUIRE(out_start[k] >= 0, "%s: item %d has out_start %lld (must be >= 0)", who, k, out_start[k]);
    DS_REQUIRE(out_lengths[k] > 0, "%s: item %d has out_length %lld (must be > 0)", who, k, out_lengths[k]);
    DS_REQUIRE(out_start[k] + out_lengths[k] <= full, "%s: item %d: out_start %lld + out_length %lld is past its full length %lld", who,
               k, out_start[k], out_lengths[k], full);
  }
  const size_t U = (size_t)B + H, n1 = (size_t)B + 1;
  p.meta.assign((U + 1) + 2 * U + n1 + 3 * (size_t)B + n1 + B, 0);
  p.foff = p.meta.data();
  p.soff = p.foff + U + 1;
  p.slen = p.soff + U;
  p.goff = p.slen + U;
  p.slo = p.goff + n1;
  p.hrow = p.slo + B;
  p.hq = p.hrow + B;
  p.ooff = p.hq + B;
  p.ostart = p.ooff + n1;
  long long xs = 0, hs = 0;
  for (size_t u = 0; u < U; ++u) {
    const long long L = u < (size_t)B ? x_lengths[u] : h_lengths[u - B];
    p.soff[u] = u < (size_t)B ? xs : hs;
    (u < (size_t)B ? xs : hs) += L;
    p.slen[u] = L;
    p.foff[u + 1] = p.foff[u] + (L + PART - 1) / PART;
  }
  for (int k = 0; k < B; ++k) {
    const long long nbx = p.foff[k + 1] - p.foff[k], Q = p.foff[B + h_index[k] + 1] - p.foff[B + h_index[k]];
    const long long lo = out_start[k] / PART - 1 > 0 ? out_start[k] / PART - 1 : 0;
    const long long hi_full = nbx + Q - 2, hi_out = (out_start[k] + out_lengths[k] - 1) / PART;
    p.slo[k] = lo;
    p.goff[k + 1] = p.goff[k] + (hi_out < hi_full ? hi_out : hi_full) - lo + 1;
    p.hrow[k] = p.foff[B + h_index[k]];
    p.hq[k] = Q;
    p.ooff[k + 1] = p.ooff[k] + out_lengths[k];
    p.ostart[k] = out_start[k];
  }
  p.n_rows = p.foff[U];
  p.n_seg = p.goff[B];
  p.n_out = p.ooff[B];
  const long long tiles = (p.n_out + OUT_TILE - 1) / OUT_TILE;
  DS_REQUIRE((p.n_rows + WPB - 1) / WPB <= INT_MAX && (p.n_seg + WPB - 1) / WPB <= INT_MAX && tiles <= INT_MAX,
             "%s: %lld spectrum rows, %lld segments, %lld outputs: too many for one call", who, p.n_rows, p.n_seg, p.n_out);
  p.n_tiles = (int)tiles;
  p.ws.stage(p.meta.data(), p.meta.size());
  p.off_spec = p.ws.reserve((size_t)p.n_rows * NBIN * sizeof(float2));
  p.off_seg = p.ws.reserve((size_t)p.n_seg * NFFT * sizeof(float));
  if (target_peak > 0.f) p.off_peak = p.ws.reserve((size_t)p.n_tiles * sizeof(float));
  return DS_OK;
}

}  // namespace
}  // namespace ds

using namespace ds;

extern "C" {

int ds_fftconvolve_workspace(const long long* x_lengths, int B, const long long* h_lengths, int H, const long long* h_index,
                             const long long* out_start, const long long* out_lengths, float target_peak, long long* bytes) {
  DS_REQUIRE(bytes, "ds_fftconvolve_workspace: bytes must be non-null");
  ConvPlan p;
  int rc = plan_conv(x_lengths, B, h_lengths, H, h_index, out_start, out_lengths, target_peak, "ds_fftconvolve_workspace", p);
  if (rc) return rc;
  *bytes = (long long)p.ws.bytes;
  return DS_OK;
}

int ds_fftconvolve(const float* d_x, const float* d_h, float* d_out, const long long* x_lengths, int B, const long long* h_lengths, int H,
                   const long long* h_index, const long long* out_start, const long long* out_lengths, int accumulate, float target_peak,
                   void* d_ws, long long ws_bytes, void* stream) {
  DS_REQUIRE(d_x && d_h && d_out && d_ws, "ds_fftconvolve: d_x, d_h, d_out and d_ws must be non-null");
  DS_REQUIRE(accumulate == 0 || accumulate == 1, "ds_fftconvolve: accumulate %d (must be 0 or 1)", accumulate);
  ConvPlan p;
  int rc = plan_conv(x_lengths, B, h_lengths, H, h_index, out_start, out_lengths, target_peak, "ds_fftconvolve", p);
  if (rc) return rc;
  DS_REQUIRE(ws_bytes >= (long long)p.ws.bytes, "ds_fftconvolve: workspace of %lld bytes, %zu needed", ws_bytes, p.ws.bytes);
  float2 *tw512, *tw1024, *tw2048;
  cudaStream_t st = (cudaStream_t)stream;
  rc = get_twiddles(st, &tw512, &tw1024, &tw2048);
  if (rc) return rc;
  uint8_t* ws = (uint8_t*)d_ws;
  const long long* m = (const long long*)ws;
  auto dev = [&](const long long* host) { return m + (host - p.meta.data()); };
  float2* spec = (float2*)(ws + p.off_spec);
  float* seg = (float*)(ws + p.off_seg);
  float* peak = target_peak > 0.f ? (float*)(ws + p.off_peak) : nullptr;
  DS_CHECK_CUDA(p.ws.upload(ws, st));
  const size_t smem = WPB * XS_PITCH * sizeof(float2);
  DS_CHECK_CUDA(cudaFuncSetAttribute(conv_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(cudaFuncSetAttribute(conv_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(launch_pdl(conv_forward_kernel, dim3((unsigned)((p.n_rows + WPB - 1) / WPB)), dim3(256), smem, st, d_x, d_h, dev(p.foff),
                           dev(p.soff), dev(p.slen), B, B + H, spec, (const float2*)tw1024, (const float2*)tw2048));
  DS_CHECK_CUDA(launch_pdl(conv_accumulate_kernel, dim3((unsigned)((p.n_seg + WPB - 1) / WPB)), dim3(256), smem, st, (const float2*)spec,
                           seg, dev(p.foff), dev(p.goff), dev(p.slo), dev(p.hrow), dev(p.hq), B, (const float2*)tw1024,
                           (const float2*)tw2048));
  DS_CHECK_CUDA(launch_pdl(conv_output_kernel, dim3((unsigned)p.n_tiles), dim3(256), (size_t)0, st, (const float*)seg, d_out, dev(p.ooff),
                           dev(p.ostart), dev(p.goff), dev(p.slo), B, accumulate, peak));
  if (peak) DS_CHECK_CUDA(launch_peak_scale(d_out, p.n_out, peak, p.n_tiles, target_peak, st));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
