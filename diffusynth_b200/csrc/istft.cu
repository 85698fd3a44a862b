// STFT+ decode fused with the inverse STFT, and the forward STFT fused with the STFT+ encode.
//   decode_stft, depad_STFT          tools.py:334-345, 185-191
//   librosa.istft(D, hop_length=256, win_length=1024) call   webUI/natural_language_guided_4/utils.py:241
//   librosa.stft(y, n_fft=1024, hop_length=256, win_length=1024) + pad_STFT + encode_stft
//                                    webUI/natural_language_guided_4/sound2sound_with_text.py:85-94; tools.py:170-182,320-331
// n_fft = 1024 (fixed by the 512 (+DC) frequency rows of the spectral representation), hop = 256,
// periodic Hann window.  Real transforms run as 512-point complex FFTs (even/odd packing), one frame per warp: radix-2
// butterflies in registers and across lanes with warp shuffles, one staging pass through shared memory for the natural-order
// result; everything is fp32 (the reference runs float64 on the CPU).
#include "common.cuh"
#include "fft_warp.cuh"
#include <mutex>
#include "../../include/diffusynth_b200.h"

namespace ds {

static constexpr int NFFT = 1024, NH = 512, HOP = 256;
static constexpr int FR = 8;   // frames per block
static constexpr int XS_PITCH = NH + NH / 16;   // staging row of a 512-point transform (fft_warp.cuh)

// ---- inverse: spec [B,3,512,T] fp32 -> windowed frames [B][T][1024] fp32; one frame per warp, FR = 8 frames per block ----
__global__ void __launch_bounds__(256)
istft_frames_kernel(const float* __restrict__ spec, float* __restrict__ frames, int T, const float2* __restrict__ tw512,
                    const float2* __restrict__ tw1024 /* e^{+2 pi i k/1024}, k<512 */) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t is_smem[];
  float2 (*X)[NH + 1] = reinterpret_cast<float2 (*)[NH + 1]>(is_smem);                                        // [FR][513]
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(is_smem + FR * (NH + 1) * sizeof(float2));   // [FR][544]
  const int b = blockIdx.y, t0 = blockIdx.x * FR;
  const float* sp = spec + (size_t)b * 3 * NH * T;
  // decode: bin f (1..512) <- row f-1 of the representation; bin 0 (DC) = 0
  for (int i = threadIdx.x; i < NH * FR; i += blockDim.x) {
    const int fr = i % FR, row = i / FR, t = t0 + fr;
    float2 v = make_float2(0.f, 0.f);
    if (t < T) {
      const float lm = __ldg(sp + (size_t)row * T + t);
      const float c = __ldg(sp + ((size_t)NH + row) * T + t), s = __ldg(sp + ((size_t)2 * NH + row) * T + t);
      const float mag = expm1f(lm);
      const float nrm = sqrtf(c * c + s * s);
      // atan2(s, c) -> (cos, sin) = (c, s)/|(c, s)|; atan2(0, 0) = 0 -> (1, 0)
      const float cc = nrm > 0.f ? c / nrm : 1.f, ss = nrm > 0.f ? s / nrm : 0.f;
      v = make_float2(mag * cc, mag * ss);
    }
    X[fr][row + 1] = v;
  }
  if (threadIdx.x < FR) X[threadIdx.x][0] = make_float2(0.f, 0.f);
  __syncthreads();
  const int fr = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Z[k] = (X[k] + conj(X[512-k])) + i * w^k * (X[k] - conj(X[512-k])),  w = e^{2 pi i/1024}; c2r ignores Im of DC/Nyquist
  float2 x[16];
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int k = lane + 32 * r;
    float2 a = X[fr][k], c = X[fr][NH - k];
    if (k == 0) { a.y = 0.f; c.y = 0.f; }
    const float2 e = make_float2(a.x + c.x, a.y - c.y);
    const float2 o = cmul(make_float2(a.x - c.x, a.y + c.y), __ldg(tw1024 + k));
    x[r] = make_float2(e.x - o.y, e.y + o.x);
  }
  fft_warp<+1, 16>(x, tw512, lane);
  store_bitrev<16>(xs[fr], x, lane);
  __syncwarp();
  // x[2n] = Re z[n] / 1024, x[2n+1] = Im z[n] / 1024; times the periodic Hann window
  const int t = t0 + fr;
  if (t >= T) return;
  for (int n = lane; n < NH; n += 32) {
    const float2 z = xs[fr][pidx<16>(n)];
    const float w0 = 0.5f - 0.5f * cospif((float)(2 * n) / 512.0f), w1 = 0.5f - 0.5f * cospif((float)(2 * n + 1) / 512.0f);
    reinterpret_cast<float2*>(frames + ((size_t)b * T + t) * NFFT)[n] = make_float2(z.x * (1.0f / NFFT) * w0, z.y * (1.0f / NFFT) * w1);
  }
}

// ---- overlap-add, window-sum-square normalisation, centre trim: wave [B][256*(T-1)] --------------
__global__ void istft_ola_kernel(const float* __restrict__ frames, float* __restrict__ wave, int T, long long out_len) {
  pdl_enter();
  const int b = blockIdx.y;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < out_len; j += (long long)gridDim.x * blockDim.x) {
    const long long jj = j + NFFT / 2;
    int t_hi = (int)(jj / HOP);
    if (t_hi > T - 1) t_hi = T - 1;
    float acc = 0.f, wss = 0.f;
    for (int t = t_hi; t >= 0 && jj - (long long)t * HOP < NFFT; --t) {
      const int m = (int)(jj - (long long)t * HOP);
      const float w = 0.5f - 0.5f * cospif((float)m / 512.0f);
      acc += __ldg(frames + ((size_t)b * T + t) * NFFT + m);
      wss = fmaf(w, w, wss);
    }
    wave[(size_t)b * out_len + j] = wss > 1.17549435e-38f ? acc / wss : acc;
  }
}

// ---- forward: wave [B][L] fp32 (zero-padded 512 each side, "constant" centre padding) -> STFT+ [B,3,512,Tpad] ----
__global__ void __launch_bounds__(256)
stft_encode_kernel(const float* __restrict__ wave, long long L, float* __restrict__ spec, int T, int Tpad, const float2* __restrict__ tw512,
                   const float2* __restrict__ tw1024) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t st_smem[];
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(st_smem);      // [FR][544]
  const int b = blockIdx.y, t0 = blockIdx.x * FR;
  const float* wv = wave + (size_t)b * L;
  {
    // one frame per warp: z[n] = x[2n] + i x[2n+1] of the windowed frame, straight into the transform's registers
    const int fr = threadIdx.x >> 5, lane = threadIdx.x & 31, t = t0 + fr;
    float2 x[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int n = lane + 32 * r;
      const long long s0 = (long long)t * HOP - NFFT / 2 + 2 * n;
      float a = 0.f, c = 0.f;
      if (t < T) {
        if (s0 >= 0 && s0 < L) a = __ldg(wv + s0);
        if (s0 + 1 >= 0 && s0 + 1 < L) c = __ldg(wv + s0 + 1);
      }
      const float w0 = 0.5f - 0.5f * cospif((float)(2 * n) / 512.0f), w1 = 0.5f - 0.5f * cospif((float)(2 * n + 1) / 512.0f);
      x[r] = make_float2(a * w0, c * w1);
    }
    fft_warp<-1, 16>(x, tw512, lane);
    store_bitrev<16>(xs[fr], x, lane);
  }
  __syncthreads();
  // X[k] = (Z[k] + conj Z[512-k])/2 - i/2 * e^{-2 pi i k/1024} (Z[k] - conj Z[512-k]),  k = 1..512 (row k-1); DC row dropped (pad_STFT)
  float* sp = spec + (size_t)b * 3 * NH * Tpad;
  for (int i = threadIdx.x; i < NH * FR; i += blockDim.x) {
    const int fr = i % FR, row = i / FR, t = t0 + fr, k = row + 1;
    if (t >= Tpad) continue;
    float lm = 0.f, co = 1.f, si = 0.f;      // padded frames: |D| = 0 -> log1p 0 = 0, angle(0) = 0 -> cos 1, sin 0
    if (t < T) {
      const float2 zk = xs[fr][pidx<16>(k & (NH - 1))], zc = xs[fr][pidx<16>((NH - k) & (NH - 1))];
      const float2 e = make_float2(0.5f * (zk.x + zc.x), 0.5f * (zk.y - zc.y));
      const float2 d = make_float2(0.5f * (zk.x - zc.x), 0.5f * (zk.y + zc.y));
      float2 w = k < NH ? __ldg(tw1024 + k) : make_float2(-1.f, 0.f);
      w.y = -w.y;
      const float2 o = cmul(d, w);            // then multiply by -i: (x, y) -> (y, -x)
      const float re = e.x + o.y, im = e.y - o.x;
      const float mag = sqrtf(re * re + im * im);
      lm = log1pf(mag);
      if (mag > 0.f) { co = re / mag; si = im / mag; }
    }
    sp[(size_t)row * Tpad + t] = lm;
    sp[((size_t)NH + row) * Tpad + t] = co;
    sp[((size_t)2 * NH + row) * Tpad + t] = si;
  }
}

// ---- Griffin-Lim phase update (librosa.griffinlim's loop body, called from tools.py:63-76,194-223 with hop 256 / win 1024) ----
// rebuilt = STFT(iSTFT(S * angles)) arrives as a spectral representation (log1p|.|, cos, sin); with momentum m
//   a = rebuilt - m/(1+m) * tprev;   angles = a / (|a| + tiny);   tprev <- rebuilt
// and the new (cos, sin) go into channels 1, 2 of the working representation whose channel 0 holds log1p(S).
__global__ void griffinlim_update_kernel(const float* __restrict__ rebuilt, float2* __restrict__ tprev, float* __restrict__ spec,
                                         float coef, int first, long long plane /* 512*T */, long long total /* B*plane */) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / plane, k = i - b * plane;
    const float* rb = rebuilt + b * 3 * plane + k;
    const float mag = expm1f(__ldg(rb));
    const float2 r = make_float2(mag * __ldg(rb + plane), mag * __ldg(rb + 2 * plane));
    float2 a = r;
    if (!first) { const float2 p = tprev[i]; a.x -= coef * p.x; a.y -= coef * p.y; }
    tprev[i] = r;
    const float d = sqrtf(a.x * a.x + a.y * a.y) + 1.17549435e-38f;
    float* sp = spec + b * 3 * plane + k;
    sp[plane] = a.x / d;
    sp[2 * plane] = a.y / d;
  }
}

// ---- tools.decode_stft / tools.encode_stft as stand-alone elementwise kernels (the numpy drop-ins of codec.py; the sampling path
// uses the fused forms above).  T = float or double: numpy computes in the precision of its input. ----
template <typename T>
__global__ void decode_stft_kernel(const T* __restrict__ enc, T* __restrict__ out, long long plane) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < plane; i += (long long)gridDim.x * blockDim.x) {
    const T mag = expm1(enc[i]);                                  // tools.py:340
    const T ph = atan2(enc[2 * plane + i], enc[plane + i]);       // :342
    T s, c;
    sincos(ph, &s, &c);
    out[2 * i] = mag * c;                                          // :344  magnitude * (cos(phase) + 1j * sin(phase))
    out[2 * i + 1] = mag * s;
  }
}
template <typename T>
__global__ void encode_stft_kernel(const T* __restrict__ D, T* __restrict__ out, long long plane) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < plane; i += (long long)gridDim.x * blockDim.x) {
    const T re = D[2 * i], im = D[2 * i + 1];
    const T ph = atan2(im, re);                                    // np.angle, tools.py:323
    T s, c;
    sincos(ph, &s, &c);
    out[i] = log1p(hypot(re, im));                                 // :322,325
    out[plane + i] = c;                                            // :327
    out[2 * plane + i] = s;                                        // :328
  }
}

__global__ void twiddle_init_kernel(float2* tw512, float2* tw1024, float2* tw2048) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 256) { double s, c; sincospi((double)i / 256.0, &s, &c); tw512[i] = make_float2((float)c, (float)s); }
  if (i < 512) { double s, c; sincospi((double)i / 512.0, &s, &c); tw1024[i] = make_float2((float)c, (float)s); }
  if (i < 1024) { double s, c; sincospi((double)i / 1024.0, &s, &c); tw2048[i] = make_float2((float)c, (float)s); }
}

struct Twiddles { float2* tw512 = nullptr; float2* tw1024 = nullptr; float2* tw2048 = nullptr; bool ready = false; };
static Twiddles g_tw[64];
static std::mutex g_tw_mutex;

// Per-device twiddle tables, built once under a mutex on a private blocking stream and synchronised before the first use, so
// the first caller's stream (or a second host thread on another stream) can never read a half-built table.  The build
// allocates, so it must not run during a stream capture: a capturing first call is refused (callers warm up once).
int get_twiddles(cudaStream_t stream, float2** a, float2** b, float2** c) {
  int dev = 0;
  DS_CHECK_CUDA(cudaGetDevice(&dev));
  DS_REQUIRE(dev >= 0 && dev < 64, "istft: device index %d out of range", dev);
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  Twiddles& t = g_tw[dev];
  if (!t.ready) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    DS_CHECK_CUDA(cudaStreamIsCapturing(stream, &cs));
    DS_REQUIRE(cs == cudaStreamCaptureStatusNone, "istft: the first STFT/iSTFT call on a device builds its twiddle tables and cannot be captured in a graph; run it once eagerly");
    DS_CHECK_CUDA(cudaMalloc(&t.tw512, 256 * sizeof(float2)));
    DS_CHECK_CUDA(cudaMalloc(&t.tw1024, 512 * sizeof(float2)));
    DS_CHECK_CUDA(cudaMalloc(&t.tw2048, 1024 * sizeof(float2)));
    cudaStream_t s0;
    DS_CHECK_CUDA(cudaStreamCreate(&s0));
    twiddle_init_kernel<<<4, 256, 0, s0>>>(t.tw512, t.tw1024, t.tw2048);
    DS_CHECK_CUDA(cudaGetLastError());
    DS_CHECK_CUDA(cudaStreamSynchronize(s0));
    DS_CHECK_CUDA(cudaStreamDestroy(s0));
    t.ready = true;
  }
  *a = t.tw512;
  *b = t.tw1024;
  *c = t.tw2048;
  return DS_OK;
}

}  // namespace ds

using namespace ds;

extern "C" {

long long ds_istft_length(int T) { return (long long)HOP * (T - 1); }

/* d_spec fp32 [B,3,512,T] (decoder output) -> d_wave fp32 [B, 256*(T-1)].  d_frames: scratch fp32 [B*T*1024]. */
int ds_stft_decode_istft(const float* d_spec, float* d_frames, float* d_wave, int B, int T, void* stream) {
  DS_REQUIRE(d_spec && d_frames && d_wave && B > 0 && T > 1, "ds_stft_decode_istft: bad arguments");
  float2 *tw512, *tw1024, *tw2048;
  int rc = get_twiddles((cudaStream_t)stream, &tw512, &tw1024, &tw2048);
  if (rc) return rc;
  const size_t smem = FR * (NH + 1) * sizeof(float2) + FR * XS_PITCH * sizeof(float2);
  DS_CHECK_CUDA(cudaFuncSetAttribute(istft_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(launch_pdl(istft_frames_kernel, dim3(dim3((T + FR - 1) / FR, B)), dim3(256), (size_t)(smem), (cudaStream_t)stream, d_spec, d_frames, T, tw512, tw1024));
  DS_CHECK_CUDA(cudaGetLastError());
  const long long out_len = ds_istft_length(T);
  DS_CHECK_CUDA(launch_pdl(istft_ola_kernel, dim3(dim3((unsigned)((out_len + 255) / 256), B)), dim3(256), (size_t)(0), (cudaStream_t)stream, d_frames, d_wave, T, out_len));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

/* d_wave fp32 [B, L] -> d_spec fp32 [B,3,512,Tpad] with T = 1 + L/256 frames, zero-padded in time to Tpad (pad_STFT). */
int ds_stft_encode(const float* d_wave, long long L, float* d_spec, int B, int Tpad, void* stream) {
  DS_REQUIRE(d_wave && d_spec && B > 0 && L > 0 && Tpad > 0, "ds_stft_encode: bad arguments");
  const int T = 1 + (int)(L / HOP);
  DS_REQUIRE(T <= Tpad, "ds_stft_encode: %d frames exceed the time resolution %d", T, Tpad);
  float2 *tw512, *tw1024, *tw2048;
  int rc = get_twiddles((cudaStream_t)stream, &tw512, &tw1024, &tw2048);
  if (rc) return rc;
  const size_t smem = FR * XS_PITCH * sizeof(float2);
  DS_CHECK_CUDA(cudaFuncSetAttribute(stft_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(launch_pdl(stft_encode_kernel, dim3(dim3((Tpad + FR - 1) / FR, B)), dim3(256), (size_t)(smem), (cudaStream_t)stream, d_wave, L, d_spec, T, Tpad, tw512, tw1024));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

/* tools.decode_stft (tools.py:334-345): d_enc [3, plane] (log1p magnitude, cos, sin) -> d_out [plane] complex (re, im interleaved);
   tools.encode_stft (:320-331): the inverse mapping.  is_double selects float64 (numpy computes in the precision of its input). */
int ds_decode_stft(const void* d_enc, void* d_out, long long plane, int is_double, void* stream) {
  DS_REQUIRE(d_enc && d_out && plane > 0, "ds_decode_stft: bad arguments");
  const unsigned blocks = grid_for(plane, 256, 16);
  if (is_double) decode_stft_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)d_enc, (double*)d_out, plane);
  else decode_stft_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)d_enc, (float*)d_out, plane);
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}
int ds_encode_stft(const void* d_D, void* d_out, long long plane, int is_double, void* stream) {
  DS_REQUIRE(d_D && d_out && plane > 0, "ds_encode_stft: bad arguments");
  const unsigned blocks = grid_for(plane, 256, 16);
  if (is_double) encode_stft_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)d_D, (double*)d_out, plane);
  else encode_stft_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)d_D, (float*)d_out, plane);
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

/* One Griffin-Lim phase update on spectral representations [B,3,512,T] (see griffinlim_update_kernel):
   d_rebuilt = ds_stft_encode(ds_stft_decode_istft(d_spec)); d_tprev fp32 [B,512,T,2] carries the previous rebuilt STFT. */
int ds_griffinlim_update(const float* d_rebuilt, float* d_tprev, float* d_spec, float momentum, int first, int B, int T, void* stream) {
  DS_REQUIRE(d_rebuilt && d_tprev && d_spec && B > 0 && T > 0 && momentum >= 0.f, "ds_griffinlim_update: bad arguments");
  const long long plane = (long long)NH * T, total = plane * B;
  const unsigned blocks = grid_for(total, 256, 16);
  griffinlim_update_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_rebuilt, reinterpret_cast<float2*>(d_tprev), d_spec,
                                                                                momentum / (1.0f + momentum), first, plane, total);
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
