// Warp-level complex FFT shared by the STFT kernels of istft.cu (n_fft 1024: 512-point complex transforms) and pitch.cu
// (n_fft 2048: 1024-point complex transforms).  One frame per warp; R points per lane.
#pragma once
#include "common.cuh"

namespace ds {

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

template <int R> struct Log2;
template <> struct Log2<16> { static constexpr int v = 4; };
template <> struct Log2<32> { static constexpr int v = 5; };

// N = 32 R point complex DFT of one frame per WARP, in registers with warp-shuffle butterflies:
//   out[n] = sum_k in[k] e^{SIGN*2*pi*i*k*n/N}.
// Lane l holds the R points i = l + 32 r (r = register index).  Radix-2 decimation in frequency: the log2(R) stages that pair
// points N/2 .. 32 apart are register-to-register, the five that pair points 16 .. 1 apart exchange registers between lanes with
// __shfl_xor_sync; no shared memory and no block barrier inside the transform.  On return x[r] holds
// out[bitrev(l + 32 r)] = out[(bitrev5(l) << log2 R) | bitrev_{log2 R}(r)].  tw: e^{+2 pi i j/N}, j < N/2.
template <int SIGN, int R>
__device__ __forceinline__ void fft_warp(float2 (&x)[R], const float2* __restrict__ tw, int lane) {
  constexpr int LR = Log2<R>::v;
#pragma unroll
  for (int rb = LR - 1; rb >= 0; --rb) {     // point-index bit b = rb + 5 lives in the register index
    const int half = 1 << rb;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (r & half) continue;
      float2 w = __ldg(tw + ((lane + 32 * (r & (half - 1))) << (LR - 1 - rb)));      // W_N^((i mod 2^b) * 2^(log2(N/2)-b))
      if (SIGN < 0) w.y = -w.y;
      const float2 u = x[r], v = x[r + half];
      x[r] = cadd(u, v);
      x[r + half] = cmul(csub(u, v), w);
    }
  }
#pragma unroll
  for (int b = 4; b >= 0; --b) {             // point-index bit b is lane bit b
    const int m = 1 << b;
    const bool upper = (lane & m) != 0;
    float2 w = __ldg(tw + ((lane & (m - 1)) << (LR + 4 - b)));
    if (SIGN < 0) w.y = -w.y;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float2 o = make_float2(__shfl_xor_sync(0xffffffffu, x[r].x, m), __shfl_xor_sync(0xffffffffu, x[r].y, m));
      x[r] = upper ? cmul(csub(o, x[r]), w) : cadd(x[r], o);
    }
  }
}

// The transform's results are staged once in shared memory in natural order, one padding entry per R (the lanes of a warp
// write bins R apart): xs[frame][pidx<R>(bin)], N + N/R entries per frame.
template <int R> __device__ __forceinline__ int pidx(int k) { return k + (k >> Log2<R>::v); }
template <int R>
__device__ __forceinline__ void store_bitrev(float2* __restrict__ xs, const float2 (&x)[R], int lane) {
  constexpr int LR = Log2<R>::v;
  const int hi = (int)(__brev((unsigned)lane) >> 27) << LR;
#pragma unroll
  for (int r = 0; r < R; ++r) xs[pidx<R>(hi | (int)(__brev((unsigned)r) >> (32 - LR)))] = x[r];
}

// ---- 2048-point real transforms from the 1024-point complex one (pitch.cu, convolve.cu) ------------------------------------
// Forward: z[n] = x[2n] + i x[2n+1] went through fft_warp<-1, R> and store_bitrev into xs; the 1025 bins of the real spectrum are
//   X[k] = (Z[k] + conj Z[1024-k])/2 - i/2 e^{-2 pi i k/2048} (Z[k] - conj Z[1024-k]),  k = 0..1024, written to out[k].
template <int R>
__device__ __forceinline__ void rfft2048_unpack(const float2* __restrict__ xs, float2* __restrict__ out, const float2* __restrict__ tw2048,
                                                int lane) {
  constexpr int NC = 32 * R;
  for (int b = lane; b < NC + 1; b += 32) {
    const float2 zk = xs[pidx<R>(b & (NC - 1))], zc = xs[pidx<R>((NC - b) & (NC - 1))];
    const float2 e = make_float2(0.5f * (zk.x + zc.x), 0.5f * (zk.y - zc.y));
    const float2 d = make_float2(0.5f * (zk.x - zc.x), 0.5f * (zk.y + zc.y));
    float2 w = b < NC ? __ldg(tw2048 + b) : make_float2(-1.f, 0.f);
    w.y = -w.y;
    const float2 o = cmul(d, w);                          // then multiply by -i: (x, y) -> (y, -x)
    out[b] = make_float2(e.x + o.y, e.y - o.x);
  }
}
// Inverse: the input of fft_warp<+1, R> at point k from the bins a = X[k] and c = X[1024-k],
//   Z[k] = (X[k] + conj X[1024-k]) + i e^{2 pi i k/2048} (X[k] - conj X[1024-k]); irfft ignores Im of DC and Nyquist (k == 0).
//   The caller scales the transform's result by 1/2048, as numpy's irfft does.
__device__ __forceinline__ float2 irfft2048_pack(float2 a, float2 c, const float2* __restrict__ tw2048, int k) {
  if (k == 0) { a.y = 0.f; c.y = 0.f; }
  const float2 e = make_float2(a.x + c.x, a.y - c.y);
  const float2 o = cmul(make_float2(a.x - c.x, a.y + c.y), __ldg(tw2048 + k));
  return make_float2(e.x - o.y, e.y + o.x);
}

// Per-device twiddle tables e^{+2 pi i j/N}, j < N/2, for N = 512, 1024 and 2048 (istft.cu).  Built on first use; that first
// call must not be under stream capture.
int get_twiddles(cudaStream_t stream, float2** tw512, float2** tw1024, float2** tw2048);

}  // namespace ds
