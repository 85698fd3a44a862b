// Image products of the decode glue (SURVEY 8a row a23 / 8f item 2), batched on the device:
//   spectrogram_to_Gradio_image (+ tools.np_power_to_db)     webUI/natural_language_guided_4/utils.py:8-50, tools.py:41-50
//   phase_to_Gradio_image                                    webUI/natural_language_guided_4/utils.py:53-91
//   latent_representation_to_Gradio_image                    webUI/natural_language_guided_4/utils.py:94-128
// taken directly from the spectral representation [B,3,512,T] (what decode_stft -> depad_STFT -> np.abs / np.angle see,
// utils.py:229-238), so the whole 6-list result of encodeBatch2GradioOutput_STFT is produced without the per-sample CPU loop.
// The reference evaluates the dB scale and the angle in float64 on complex128 data; so do these kernels (fp64 is a tiny
// share of the work: 131 k bins per timbre); the complex bin itself is the fp32 product the iSTFT kernel uses.
// All three are HBM-bound byte producers: 12 bytes read + 6 bytes written per bin (two passes read the representation twice).
#include "common.cuh"
#include "../../include/diffusynth_b200.h"

namespace ds {

static constexpr int IM_NH = 512;

// fp32 complex bin of representation row `row` (bin row+1), exactly as istft_frames_kernel decodes it
__device__ __forceinline__ float2 decode_bin(const float* __restrict__ sp, int T, int row, int t) {
  const float lm = __ldg(sp + (size_t)row * T + t);
  const float c = __ldg(sp + ((size_t)IM_NH + row) * T + t), s = __ldg(sp + ((size_t)2 * IM_NH + row) * T + t);
  const float mag = expm1f(lm);
  const float nrm = sqrtf(c * c + s * s);
  const float cc = nrm > 0.f ? c / nrm : 1.f, ss = nrm > 0.f ? s / nrm : 0.f;
  return make_float2(mag * cc, mag * ss);
}

__device__ __forceinline__ double bin_abs(float2 v) { return hypot((double)v.x, (double)v.y); }

// numpy's float64 -> uint8 cast on x86-64: truncate to a (32-bit) integer, keep the low byte; NaN -> 0
__device__ __forceinline__ unsigned char cast_u8(double v) {
  if (!(v == v)) return 0;
  return (unsigned char)((int)v & 0xff);
}

// ---- pass 1: per-sample maximum of |D| (np_power_to_db's `ref = S.max()`); non-negative doubles order like their bits ----
__global__ void __launch_bounds__(256)
spec_absmax_kernel(const float* __restrict__ spec, unsigned long long* __restrict__ absmax, int T) {
  const int b = blockIdx.y;
  const float* sp = spec + (size_t)b * 3 * IM_NH * T;
  const long long total = (long long)IM_NH * T;
  double m = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / T), t = (int)(i - (long long)row * T);
    const double a = bin_abs(decode_bin(sp, T, row, t));
    if (a > m) m = a;            // NaN never wins, like np.max would not be reproduced anyway
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_xor_sync(0xffffffffu, m, o);
    m = other > m ? other : m;
  }
  __shared__ double s_m[8];
  if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = s_m[w] > m ? s_m[w] : m;
    atomicMax(absmax + b, (unsigned long long)__double_as_longlong(m));
  }
}

// ---- pass 2: the two uint8 [513, T, 3] renderings, flipped vertically (image row r shows bin 512 - r; bin 0 is the zero DC row) ----
__global__ void __launch_bounds__(256)
spec_images_kernel(const float* __restrict__ spec, const unsigned long long* __restrict__ absmax,
                   unsigned char* __restrict__ mag_img, unsigned char* __restrict__ phase_img, int T) {
  const int b = blockIdx.y;
  const float* sp = spec + (size_t)b * 3 * IM_NH * T;
  const long long total = (long long)(IM_NH + 1) * T;
  const double ref = __longlong_as_double((long long)absmax[b]);
  // np_power_to_db (tools.py:41-50) with np_log10(x) = log(x + 1e-16) / log(10) (tools.py:11-15)
  const double db_ref = 10.0 * (log(fmax(1e-16, ref) + 1e-16) / log(10.0));
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / T), t = (int)(i - (long long)r * T);
    const int bin = IM_NH - r;
    double S = 0.0, ph = 0.0;
    if (bin > 0) {
      const float2 v = decode_bin(sp, T, bin - 1, t);
      S = bin_abs(v);
      ph = atan2((double)v.y, (double)v.x);
    }
    double db = 10.0 * (log(fmax(1e-16, S) + 1e-16) / log(10.0)) - db_ref;
    db = fmax(db, 0.0 - 80.0);                 // log_spec.max() is the reference bin itself: db_ref - db_ref = 0
    const unsigned char g = cast_u8(255.0 * ((db + 80.0) / 80.0));
    const unsigned char p = cast_u8(255.0 * ((ph + 1.0) / 2.0));
    unsigned char* mo = mag_img + ((size_t)b * (IM_NH + 1) * T + i) * 3;
    unsigned char* po = phase_img + ((size_t)b * (IM_NH + 1) * T + i) * 3;
    mo[0] = g; mo[1] = g; mo[2] = 63;          // 255 * ((-60 + 80) / 80) = 63.75
    po[0] = p; po[1] = p; po[2] = 51;          // 255 * 0.2 = 51.0
  }
}

// ---- latent image: per-(sample, channel) min / max, then [8H, 8W, 4] uint8, flipped vertically -------------------------
__global__ void __launch_bounds__(256)
latent_minmax_kernel(const float* __restrict__ lat, float2* __restrict__ mm, long long hw) {
  const float* p = lat + (size_t)blockIdx.x * hw;
  float lo = INFINITY, hi = -INFINITY;
  for (long long i = threadIdx.x; i < hw; i += blockDim.x) {
    const float v = __ldg(p + i);
    lo = fminf(lo, v);
    hi = fmaxf(hi, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  __shared__ float s_lo[8], s_hi[8];
  if ((threadIdx.x & 31) == 0) { s_lo[threadIdx.x >> 5] = lo; s_hi[threadIdx.x >> 5] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { lo = fminf(lo, s_lo[w]); hi = fmaxf(hi, s_hi[w]); }
    mm[blockIdx.x] = make_float2(lo, hi);
  }
}

// thread = (sample, output row, source column): 8 identical RGBA pixels = 32 contiguous bytes
__global__ void __launch_bounds__(256)
latent_image_kernel(const float* __restrict__ lat, const float2* __restrict__ mm, unsigned char* __restrict__ img, int B, int H, int W) {
  const long long total = (long long)B * 8 * H * W;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % W);
    const long long r = i / W;
    const int yo = (int)(r % (8 * H)), b = (int)(r / (8 * H));
    const int y = (8 * H - 1 - yo) >> 3;        // np.flipud of the 8x row-repeated image
    uint32_t px = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float2 m = __ldg(mm + b * 4 + c);
      const float v = __ldg(lat + (((size_t)b * 4 + c) * H + y) * W + x);
      // ((img - min) / (max - min) * 255) in float32, then astype(uint8): truncation; 0/0 = NaN -> 0
      const float q = __fmul_rn(__fdiv_rn(__fsub_rn(v, m.x), __fsub_rn(m.y, m.x)), 255.0f);
      const uint32_t u = (q == q) ? (uint32_t)((int)q & 0xff) : 0u;
      px |= u << (8 * c);
    }
    uint4* o = reinterpret_cast<uint4*>(img + (((size_t)b * 8 * H + yo) * 8 * W + (size_t)8 * x) * 4);
    o[0] = make_uint4(px, px, px, px);
    o[1] = make_uint4(px, px, px, px);
  }
}

}  // namespace ds

using namespace ds;

extern "C" {

/* d_spec fp32 [B,3,512,T] -> d_mag_img, d_phase_img uint8 [B,513,T,3]; d_absmax: scratch, 8 bytes per sample. */
int ds_spec_images(const float* d_spec, void* d_mag_img, void* d_phase_img, void* d_absmax, int B, int T, void* stream) {
  DS_REQUIRE(d_spec && d_mag_img && d_phase_img && d_absmax && B > 0 && T > 0, "ds_spec_images: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  DS_CHECK_CUDA(cudaMemsetAsync(d_absmax, 0, (size_t)B * 8, st));
  const long long bins = (long long)IM_NH * T;
  int gx = (int)((bins + 256 * 4 - 1) / (256 * 4));
  if (gx < 1) gx = 1;
  spec_absmax_kernel<<<dim3(gx, B), 256, 0, st>>>(d_spec, reinterpret_cast<unsigned long long*>(d_absmax), T);
  DS_CHECK_CUDA(cudaGetLastError());
  const long long px = (long long)(IM_NH + 1) * T;
  spec_images_kernel<<<dim3((unsigned)((px + 255) / 256), B), 256, 0, st>>>(d_spec, reinterpret_cast<const unsigned long long*>(d_absmax),
                                                                            reinterpret_cast<unsigned char*>(d_mag_img),
                                                                            reinterpret_cast<unsigned char*>(d_phase_img), T);
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

/* d_lat fp32 [B,4,H,W] -> d_img uint8 [B,8H,8W,4]; d_minmax: scratch, 8 bytes per (sample, channel). */
int ds_latent_image(const float* d_lat, void* d_img, void* d_minmax, int B, int H, int W, void* stream) {
  DS_REQUIRE(d_lat && d_img && d_minmax && B > 0 && H > 0 && W > 0, "ds_latent_image: bad arguments");
  DS_REQUIRE(reinterpret_cast<uintptr_t>(d_img) % 16 == 0, "ds_latent_image: the image must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  latent_minmax_kernel<<<B * 4, 256, 0, st>>>(d_lat, reinterpret_cast<float2*>(d_minmax), (long long)H * W);
  DS_CHECK_CUDA(cudaGetLastError());
  const long long total = (long long)B * 8 * H * W;
  latent_image_kernel<<<grid_for(total, 256, 32), 256, 0, st>>>(d_lat, reinterpret_cast<const float2*>(d_minmax), reinterpret_cast<unsigned char*>(d_img), B, H, W);
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
