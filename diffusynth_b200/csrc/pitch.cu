// Pitch shifting and track mixing for note arrangements (track_maker.DiffSynth after the per-note closure, track_maker.py:42):
//   librosa.effects.pitch_shift(y, sr=16000, n_steps=n, bins_per_octave=12) with librosa's default STFT arguments
//     = time_stretch(y, rate = 2^(-n/12)) -> resample(16000/rate -> 16000 Hz) -> fix_length(len(y)),
//     time_stretch = stft(n_fft 2048, hop 512, periodic Hann, centre zero padding) -> phase_vocoder(hop 512)
//                    -> istft(length = round(len(y)/rate));
//   then every note is scaled by its gain, placed at its onset and summed into one track.
// The resampler is a Kaiser-windowed sinc evaluated directly (resampy's kaiser_best parameters), not librosa's default soxr
// (DESIGN.md section 8).  Every stage runs over a ragged batch: per-item prefix offsets into packed buffers, lengths and rates as
// plain device arrays, one launch per stage whatever the number of items.  Everything is fp32 except the positions and the
// rates, which are float64 like numpy's.
#include "common.cuh"
#include "fft_warp.cuh"
#include <cmath>
#include <type_traits>
#include <vector>
#include "../../include/diffusynth_b200.h"

namespace ds {
namespace {

constexpr int NFFT = 2048, NC = 1024 /* complex points */, NBIN = NFFT / 2 + 1, HOP = 512;
constexpr int R = NC / 32;                      // points per lane
constexpr int XS_PITCH = NC + NC / R;           // staging row (fft_warp.cuh)
constexpr int FR = 8;                           // frames (warps) per block
constexpr int MIX_TILE = 1024;                  // track samples per mix block

__device__ __forceinline__ float hann2048(int m) { return 0.5f - 0.5f * cospif((float)m / 1024.0f); }

// ---- forward STFT: y (packed, item k at loff[k], length L_k) -> D [frames][1025] complex; one frame per warp ----------------
// frame t of item k covers samples t*512 - 1024 .. t*512 + 1023 (centre zero padding); z[n] = x[2n] + i x[2n+1] of the windowed
// frame goes through one 1024-point complex FFT, the real spectrum is unpacked from it.
__global__ void __launch_bounds__(256)
pitch_stft_kernel(const float* __restrict__ y, const long long* __restrict__ loff, const long long* __restrict__ fin, int B,
                  float2* __restrict__ D, const float2* __restrict__ tw1024, const float2* __restrict__ tw2048) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t ps_smem[];
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(ps_smem);
  const int fr = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long g = (long long)blockIdx.x * FR + fr;
  if (g >= __ldg(fin + B)) return;                       // whole warps leave: the transform is warp-local
  const int k = find_item(fin, B, g);
  const long long t = g - __ldg(fin + k), L = __ldg(loff + k + 1) - __ldg(loff + k);
  const float* wv = y + __ldg(loff + k);
  float2 x[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int n = lane + 32 * r;
    const long long s0 = t * HOP - NFFT / 2 + 2 * n;
    const float a = (s0 >= 0 && s0 < L) ? __ldg(wv + s0) : 0.f;
    const float c = (s0 + 1 >= 0 && s0 + 1 < L) ? __ldg(wv + s0 + 1) : 0.f;
    x[r] = make_float2(a * hann2048(2 * n), c * hann2048(2 * n + 1));
  }
  fft_warp<-1, R>(x, tw1024, lane);
  store_bitrev<R>(xs[fr], x, lane);
  __syncwarp();
  rfft2048_unpack<R>(xs[fr], D + g * NBIN, tw2048, lane);
}

// ---- phase vocoder (librosa.phase_vocoder, hop 512): one thread per (item, bin), output frames walked in order ----------------
// step_t = t * rate (float64, numpy's arange); |S| interpolates |D| linearly between frames floor(step) and floor(step)+1 (D
// zero-padded by two frames); the phase accumulator starts at angle(D[0]) and advances by phi + wrap(dphase - phi).  It is kept
// wrapped to [-pi, pi): unwrapped it grows to ~1e5 rad, where an fp32 ulp is ~0.008 rad.  phi = bin * pi * hop / 1024 is
// reduced mod 2 pi in float64.
__device__ __forceinline__ float wrap_pi(float v) {           // x - 2 pi round(x / 2 pi), numpy's rounding (half to even)
  return v - 6.283185307179586f * rintf(v * 0.15915494309189535f);
}
__global__ void __launch_bounds__(256)
pitch_vocoder_kernel(const float2* __restrict__ D, float2* __restrict__ S, const long long* __restrict__ fin,
                     const long long* __restrict__ fout, const double* __restrict__ rate, int B) {
  pdl_enter();
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)B * NBIN) return;
  const int k = (int)(gid / NBIN), bin = (int)(gid - (long long)k * NBIN);
  const long long f0 = __ldg(fin + k), T_in = __ldg(fin + k + 1) - f0, o0 = __ldg(fout + k), T_out = __ldg(fout + k + 1) - o0;
  const double rt = __ldg(rate + k);
  double adv = fmod((double)bin * (kPi * HOP / (NFFT / 2)), 2.0 * kPi);
  if (adv >= kPi) adv -= 2.0 * kPi;
  const float phi = (float)adv;
  const float2* Dk = D + f0 * NBIN + bin;
  float2* Sk = S + o0 * NBIN + bin;
  float2 c0 = __ldg(Dk);
  float acc = atan2f(c0.y, c0.x);
  for (long long t = 0; t < T_out; ++t) {
    const double step = (double)t * rt;
    const long long i = (long long)floor(step);
    const float a = (float)(step - (double)i);
    c0 = __ldg(Dk + i * NBIN);
    const float2 c1 = i + 1 < T_in ? __ldg(Dk + (i + 1) * NBIN) : make_float2(0.f, 0.f);
    const float mag = (1.0f - a) * hypotf(c0.x, c0.y) + a * hypotf(c1.x, c1.y);
    float sn, cs;
    sincosf(acc, &sn, &cs);
    Sk[t * NBIN] = make_float2(mag * cs, mag * sn);
    const float dph = wrap_pi(atan2f(c1.y, c1.x) - atan2f(c0.y, c0.x) - phi);
    acc = acc + phi + dph;
    acc -= 6.283185307179586f * floorf((acc + 3.14159265358979f) * 0.15915494309189535f);     // back to [-pi, pi)
  }
}

// ---- inverse STFT frames: S [frames][1025] -> windowed frames [frames][2048]; one frame per warp -------------------------------
__global__ void __launch_bounds__(256)
pitch_istft_frames_kernel(const float2* __restrict__ S, float* __restrict__ frames, long long n_frames,
                          const float2* __restrict__ tw1024, const float2* __restrict__ tw2048) {
  pdl_enter();
  extern __shared__ __align__(16) uint8_t pi_smem[];
  float2 (*xs)[XS_PITCH] = reinterpret_cast<float2 (*)[XS_PITCH]>(pi_smem);
  const int fr = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long g = (long long)blockIdx.x * FR + fr;
  if (g >= n_frames) return;
  const float2* X = S + g * NBIN;
  float2 x[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int k = lane + 32 * r;
    x[r] = irfft2048_pack(__ldg(X + k), __ldg(X + NC - k), tw2048, k);
  }
  fft_warp<+1, R>(x, tw1024, lane);
  store_bitrev<R>(xs[fr], x, lane);
  __syncwarp();
  float2* out = reinterpret_cast<float2*>(frames + g * NFFT);
  for (int n = lane; n < NC; n += 32) {
    const float2 z = xs[fr][pidx<R>(n)];
    out[n] = make_float2(z.x * (1.0f / NFFT) * hann2048(2 * n), z.y * (1.0f / NFFT) * hann2048(2 * n + 1));
  }
}

// ---- overlap-add with librosa's `length`: ys_k[j] = OLA / window-sum-square at j + 1024 over the first tcap[k] frames (zero past
// the overlap-added extent); item k at yoff[k], length round(L_k / rate_k) --------------------------------------------------------
__global__ void pitch_ola_kernel(const float* __restrict__ frames, float* __restrict__ ys, const long long* __restrict__ fout,
                                 const long long* __restrict__ yoff, const long long* __restrict__ tcap, int B) {
  pdl_enter();
  const long long total = __ldg(yoff + B);
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int k = find_item(yoff, B, g);
    const long long jj = g - __ldg(yoff + k) + NFFT / 2;
    const float* fk = frames + __ldg(fout + k) * NFFT;
    long long t = jj / HOP;
    const long long tc = __ldg(tcap + k);
    if (t > tc - 1) t = tc - 1;
    float acc = 0.f, wss = 0.f;
    for (; t >= 0 && jj - t * HOP < NFFT; --t) {
      const int m = (int)(jj - t * HOP);
      const float w = hann2048(m);
      acc += __ldg(fk + t * NFFT + m);
      wss = fmaf(w, w, wss);
    }
    ys[g] = wss > 1.17549435e-38f ? acc / wss : acc;
  }
}

// ---- resample 16000/rate -> 16000 Hz + fix_length: out_k[j] = sum_i ys_k[i] h(i - j/rate) for j < nval[k], zero after ------------
// h(d) = s * roll * sinc(s * roll * d) * I0(beta sqrt(1 - (s d / 64)^2)) / I0(beta), |d| <= 64 / s, s = min(1, rate); samples
// outside [0, len) count as zero.  rate == 1 (n_steps 0) copies: librosa.resample returns its input when the rates are equal.
__global__ void __launch_bounds__(256)
pitch_resample_kernel(const float* __restrict__ ys, float* __restrict__ out, const long long* __restrict__ loff,
                      const long long* __restrict__ yoff, const long long* __restrict__ nval, const double* __restrict__ rate, int B,
                      float inv_i0_beta) {
  pdl_enter();
  const long long total = __ldg(loff + B);
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int k = find_item(loff, B, g);
    const long long j = g - __ldg(loff + k);
    const float* src = ys + __ldg(yoff + k);
    const long long len = __ldg(yoff + k + 1) - __ldg(yoff + k);
    const double rt = __ldg(rate + k);
    float acc = 0.f;
    if (j < __ldg(nval + k)) {
      if (rt == 1.0) {
        acc = __ldg(src + j);
      } else {
        const double pos = (double)j / rt, sc = rt < 1.0 ? rt : 1.0, half = RS_ZEROS / sc;
        const double i0d = floor(pos);
        const long long ip = (long long)i0d;
        const float f = (float)(pos - i0d);
        long long lo = (long long)ceil(pos - half), hi = (long long)floor(pos + half);
        if (lo < 0) lo = 0;
        if (hi > len - 1) hi = len - 1;
        const float cut = (float)(sc * RS_ROLLOFF), wscale = (float)(sc / RS_ZEROS);
        for (long long i = lo; i <= hi; ++i) {
          const float d = (float)(i - ip) - f;
          const float u = d * wscale;
          const float win = cyl_bessel_i0f((float)RS_BETA * sqrtf(fmaxf(0.f, 1.0f - u * u))) * inv_i0_beta;
          const float z = cut * d;
          const float sinc = z == 0.f ? 1.f : sinpif(z) / (3.14159265358979f * z);
          acc = fmaf(__ldg(src + i), cut * sinc * win, acc);
        }
      }
    }
    out[g] = acc;
  }
}

// ---- track mix (ds_mix_arrangement, ds_mix_stereo, and ds_mix_track without fades or peak): channel c of the output, planar
// [CH][track_len], is out_c[j] = sum over notes n covering j, in input order, of gain_n,c * env_n * src[src_off_n + j - onset_n].
// A gather over track samples (one block per MIX_TILE samples) through the per-tile note lists, so the sum order is fixed.  env_n
// is a linear fade over the last fade_n = min(fade_out[n], len[n]) samples (clamped on the host); a sample before the ramp takes a
// plain fmaf(gain, src, acc), so a fade-free note has no envelope multiply at all.  When `peak` is non-null, each tile also writes
// its max |out| partial over every channel.  Every thread owns ARR_SPT samples 256 apart and walks the tile's notes once for all
// of them (a note's metadata is loaded once per thread, not once per sample); each sample still sums its notes in input order.
// CH = 1 takes one fp32 gain per note, CH = 2 one float2 (left, right) from plan_mix's pan law.  256 threads per block.
constexpr int ARR_SPT = MIX_TILE / 256;
template <int CH> using MixGain = std::conditional_t<CH == 1, float, float2>;
__device__ __forceinline__ void gain_channels(float v, float (&g)[1]) { g[0] = v; }
__device__ __forceinline__ void gain_channels(float2 v, float (&g)[2]) { g[0] = v.x; g[1] = v.y; }

template <int CH>
__global__ void __launch_bounds__(256)
pitch_arrange_kernel(const float* __restrict__ src, float* __restrict__ track, long long track_len, const int* __restrict__ tile_ptr,
                     const int* __restrict__ tile_notes, const long long* __restrict__ src_off, const long long* __restrict__ len,
                     const long long* __restrict__ onset, const MixGain<CH>* __restrict__ gain, const long long* __restrict__ fade,
                     float* __restrict__ peak) {
  pdl_enter();
  __shared__ float red[8];
  const int p0 = __ldg(tile_ptr + blockIdx.x), p1 = __ldg(tile_ptr + blockIdx.x + 1);
  const long long j0 = (long long)blockIdx.x * MIX_TILE + threadIdx.x;
  float acc[CH][ARR_SPT];
#pragma unroll
  for (int c = 0; c < CH; ++c)
#pragma unroll
    for (int k = 0; k < ARR_SPT; ++k) acc[c][k] = 0.f;
  for (int p = p0; p < p1; ++p) {
    const int n = __ldg(tile_notes + p);
    const long long on = __ldg(onset + n), L = __ldg(len + n), F = __ldg(fade + n);   // (samples past track_len have r >= L)
    float g[CH];
    gain_channels(__ldg(gain + n), g);
    const float* sn = src + __ldg(src_off + n);
#pragma unroll
    for (int k = 0; k < ARR_SPT; ++k) {
      const long long r = j0 + 256 * k - on;
      if (r < 0 || r >= L) continue;
      const float s = __ldg(sn + r);
      const long long left = L - r;                                       // 1 on the note's last sample
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        if (left > F) acc[c][k] = fmaf(g[c], s, acc[c][k]);
        else acc[c][k] = fmaf(g[c] * ((float)left / (float)F), s, acc[c][k]);
      }
    }
  }
  float pk = 0.f;
#pragma unroll
  for (int k = 0; k < ARR_SPT; ++k) {
    const long long j = j0 + 256 * k;
    if (j < track_len) {
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        track[c * track_len + j] = acc[c][k];
        pk = fmaxf(pk, fabsf(acc[c][k]));
      }
    }
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

// ---- peak normalisation: every block reduces the n_tiles partials (a maximum: exact in any order), then scales its grid-stride
// share of the track by target / max in place (both channels of a stereo mix: track_len is 2 * its length, one common scale).  An
// all-zero track stays zero.
__global__ void __launch_bounds__(512)
pitch_peak_scale_kernel(float* __restrict__ track, long long track_len, const float* __restrict__ peak, int n_tiles, float target) {
  pdl_enter();
  __shared__ float red[16];
  float m = 0.f;
  for (int t = threadIdx.x; t < n_tiles; t += blockDim.x) m = fmaxf(m, __ldg(peak + t));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  m = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, red[w]);
  if (m == 0.f) return;
  const float sc = target / m;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < track_len; j += (long long)gridDim.x * blockDim.x)
    track[j] *= sc;
}

// I0(x) by its power series sum ((x/2)^k / k!)^2 (converged to double precision for the beta used here)
double bessel_i0(double x) {
  double term = 1.0, sum = 1.0;
  for (int k = 1; k < 200 && term > 1e-17 * sum; ++k) {
    term *= (x / (2.0 * k)) * (x / (2.0 * k));
    sum += term;
  }
  return sum;
}

// Host-side plan of one batched pitch shift: the per-item metadata, staged at the start of the workspace, and the stages after
// it.  Metadata: loff, fin, fout, yoff (B+1 prefix arrays each), tcap, nval (B each) in one int64 array, then rate (B) float64.
struct PitchPlan {
  std::vector<long long> idx;
  std::vector<double> rate;
  Workspace ws;
  size_t off_idx = 0, off_rate = 0, off_D = 0, off_S = 0, off_frames = 0, off_ys = 0;
  long long n_in_frames = 0, n_out_frames = 0, n_ys = 0, n_samples = 0;
};

int plan_pitch(const long long* lengths, const double* n_steps, int B, const char* who, PitchPlan& p) {
  DS_REQUIRE(lengths && n_steps && B > 0, "%s: lengths and n_steps must be non-null and B > 0 (B = %d)", who, B);
  for (int k = 0; k < B; ++k) {
    DS_REQUIRE(lengths[k] > 0, "%s: item %d has length %lld (must be > 0)", who, k, lengths[k]);
    DS_REQUIRE(std::isfinite(n_steps[k]) && std::fabs(n_steps[k]) <= 24.0, "%s: item %d has n_steps %g (must be finite, |n_steps| <= 24)",
               who, k, n_steps[k]);
  }
  const size_t n1 = (size_t)B + 1;
  p.idx.assign(4 * n1 + 2 * (size_t)B, 0);
  p.rate.assign(B, 0.0);
  long long *loff = p.idx.data(), *fin = loff + n1, *fout = fin + n1, *yoff = fout + n1, *tcap = yoff + n1, *nval = tcap + B;
  for (int k = 0; k < B; ++k) {
    const long long L = lengths[k];
    const double rt = std::exp2(-n_steps[k] / 12.0);
    const long long T_in = 1 + L / HOP;
    const long long T_out = (long long)std::ceil((double)T_in / rt);              // len(np.arange(0, T_in, rate))
    const long long len = (long long)std::nearbyint((double)L / rt);             // round(L / rate), half to even like Python
    long long cap = (long long)std::ceil((double)(len + NFFT) / HOP);            // librosa.istft: frames needed for `length`
    if (cap > T_out) cap = T_out;
    long long nv = L;
    if (rt != 1.0) {
      const long long n_out = (long long)std::ceil((double)len * rt);            // librosa.resample output length
      if (n_out < nv) nv = n_out;
    }
    loff[k + 1] = loff[k] + L;
    fin[k + 1] = fin[k] + T_in;
    fout[k + 1] = fout[k] + T_out;
    yoff[k + 1] = yoff[k] + len;
    tcap[k] = cap;
    nval[k] = nv;
    p.rate[k] = rt;
  }
  p.n_samples = loff[B];
  p.n_in_frames = fin[B];
  p.n_out_frames = fout[B];
  p.n_ys = yoff[B];
  p.off_idx = p.ws.stage(p.idx.data(), p.idx.size());
  p.off_rate = p.ws.stage(p.rate.data(), p.rate.size());
  p.off_D = p.ws.reserve((size_t)p.n_in_frames * NBIN * sizeof(float2));
  p.off_S = p.ws.reserve((size_t)p.n_out_frames * NBIN * sizeof(float2));
  p.off_frames = p.ws.reserve((size_t)p.n_out_frames * NFFT * sizeof(float));
  p.off_ys = p.ws.reserve((size_t)p.n_ys * sizeof(float));
  return DS_OK;
}

// Per-tile note lists of a mix (CSR over tiles of MIX_TILE track samples, notes in input order) and the clamped fades, staged with
// the per-note arrays; one peak partial per tile after them when normalising.  A stereo mix stages its (left, right) gains in
// place of the fp32 gains.
struct MixPlan {
  std::vector<int> tile_ptr, tile_notes;
  std::vector<long long> fade;
  std::vector<float2> gain2;
  Workspace ws;
  size_t off_notes = 0, off_src = 0, off_len = 0, off_onset = 0, off_gain = 0, off_fade = 0, off_peak = 0;
  int n_tiles = 0;
};

// Constant-power pan law, cos(pi u / 4) for u = 1 + p (left) or 1 - p (right), in float64; cos(pi / 2) is 6.1e-17 in float64,
// so u == 2 (a hard pan) is exactly 0 and leaks nothing into the other channel.
double pan_cos(double u) { return u == 2.0 ? 0.0 : std::cos(kPi * u / 4.0); }

// The mix's checks and plan; ds_mix_track comes here with all-zero fades and target_peak 0, and only ds_mix_stereo(_workspace)
// passes pans.  src_offsets and gains are null in the workspace queries, which do not take them.
int plan_mix(const long long* src_offsets, const long long* lengths, const long long* onsets, const float* gains, const float* pans,
             const long long* fade_out, int K, float target_peak, long long track_len, const char* who, MixPlan& p) {
  DS_REQUIRE(lengths && onsets && K > 0 && track_len > 0, "%s: lengths and onsets must be non-null, K > 0 and track_len > 0", who);
  DS_REQUIRE(std::isfinite(target_peak) && target_peak >= 0.f, "%s: target_peak %g (must be finite and >= 0)", who, (double)target_peak);
  for (int n = 0; n < K; ++n) {
    DS_REQUIRE(lengths[n] > 0, "%s: note %d has length %lld (must be > 0)", who, n, lengths[n]);
    DS_REQUIRE(onsets[n] >= 0, "%s: note %d has onset %lld (must be >= 0)", who, n, onsets[n]);
    DS_REQUIRE(onsets[n] + lengths[n] <= track_len, "%s: note %d ends at %lld, past the track length %lld", who, n,
               onsets[n] + lengths[n], track_len);
    DS_REQUIRE(fade_out[n] >= 0, "%s: note %d has fade_out %lld (must be >= 0)", who, n, fade_out[n]);
    DS_REQUIRE(!src_offsets || src_offsets[n] >= 0, "%s: note %d has source offset %lld (must be >= 0)", who, n,
               src_offsets ? src_offsets[n] : 0LL);
    DS_REQUIRE(!pans || (std::isfinite(pans[n]) && std::fabs(pans[n]) <= 1.f), "%s: note %d has pan %g (must be finite, |pan| <= 1)",
               who, n, pans ? (double)pans[n] : 0.0);
  }
  p.n_tiles = (int)((track_len + MIX_TILE - 1) / MIX_TILE);
  std::vector<int> count(p.n_tiles + 1, 0);
  for (int n = 0; n < K; ++n)
    for (long long t = onsets[n] / MIX_TILE; t <= (onsets[n] + lengths[n] - 1) / MIX_TILE; ++t) ++count[t + 1];
  p.tile_ptr.assign(p.n_tiles + 1, 0);
  for (int t = 0; t < p.n_tiles; ++t) p.tile_ptr[t + 1] = p.tile_ptr[t] + count[t + 1];
  p.tile_notes.assign(p.tile_ptr[p.n_tiles], 0);
  std::vector<int> fill(p.tile_ptr.begin(), p.tile_ptr.end() - 1);
  for (int n = 0; n < K; ++n)                                 // ascending n: every tile's list is in input order
    for (long long t = onsets[n] / MIX_TILE; t <= (onsets[n] + lengths[n] - 1) / MIX_TILE; ++t) p.tile_notes[fill[t]++] = n;
  p.fade.resize(K);
  for (int n = 0; n < K; ++n) p.fade[n] = fade_out[n] < lengths[n] ? fade_out[n] : lengths[n];
  p.ws.stage(p.tile_ptr.data(), p.tile_ptr.size());
  p.off_notes = p.ws.stage(p.tile_notes.data(), p.tile_notes.size());
  p.off_src = p.ws.stage(src_offsets, K);
  p.off_len = p.ws.stage(lengths, K);
  p.off_onset = p.ws.stage(onsets, K);
  if (pans) {
    p.gain2.assign(K, make_float2(0.f, 0.f));
    for (int n = 0; gains && n < K; ++n)        // gL = g cos(pi (1 + p) / 4), gR = g cos(pi (1 - p) / 4), rounded once
      p.gain2[n] = make_float2((float)(gains[n] * pan_cos(1.0 + pans[n])), (float)(gains[n] * pan_cos(1.0 - pans[n])));
    p.off_gain = p.ws.stage(p.gain2.data(), K);
  } else {
    p.off_gain = p.ws.stage(gains, K);
  }
  p.off_fade = p.ws.stage(p.fade.data(), K);
  if (target_peak > 0.f) p.off_peak = p.ws.reserve((size_t)p.n_tiles * sizeof(float));
  return DS_OK;
}

int mix_workspace(const long long* lengths, const long long* onsets, const long long* fade_out, const float* pans, int K,
                  float target_peak, long long track_len, long long* bytes, const char* who) {
  MixPlan p;
  int rc = plan_mix(nullptr, lengths, onsets, nullptr, pans, fade_out, K, target_peak, track_len, who, p);
  if (rc) return rc;
  *bytes = (long long)p.ws.bytes;
  return DS_OK;
}

template <int CH>
cudaError_t launch_arrange(const MixPlan& p, const float* d_src, float* d_out, long long track_len, const uint8_t* ws, float* peak,
                           cudaStream_t st) {
  return launch_pdl(pitch_arrange_kernel<CH>, dim3((unsigned)p.n_tiles), dim3(256), (size_t)0, st, d_src, d_out, track_len,
                    (const int*)ws, (const int*)(ws + p.off_notes), (const long long*)(ws + p.off_src), (const long long*)(ws + p.off_len),
                    (const long long*)(ws + p.off_onset), (const MixGain<CH>*)(ws + p.off_gain), (const long long*)(ws + p.off_fade),
                    peak);
}

// d_out: [track_len] mono, or planar [2][track_len] when pans is non-null
int mix(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets, const float* gains,
        const float* pans, const long long* fade_out, int K, float target_peak, float* d_out, long long track_len, void* d_ws,
        long long ws_bytes, void* stream, const char* who) {
  MixPlan p;
  int rc = plan_mix(src_offsets, lengths, onsets, gains, pans, fade_out, K, target_peak, track_len, who, p);
  if (rc) return rc;
  DS_REQUIRE(ws_bytes >= (long long)p.ws.bytes, "%s: workspace of %lld bytes, %zu needed", who, ws_bytes, p.ws.bytes);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)d_ws;
  float* peak = target_peak > 0.f ? (float*)(ws + p.off_peak) : nullptr;
  DS_CHECK_CUDA(p.ws.upload(ws, st));
  DS_CHECK_CUDA(pans ? launch_arrange<2>(p, d_src, d_out, track_len, ws, peak, st)
                     : launch_arrange<1>(p, d_src, d_out, track_len, ws, peak, st));
  if (peak) DS_CHECK_CUDA(launch_peak_scale(d_out, (pans ? 2 : 1) * track_len, peak, p.n_tiles, target_peak, st));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // namespace

cudaError_t launch_peak_scale(float* d_out, long long n, const float* peak, int n_tiles, float target, cudaStream_t st) {
  return launch_pdl(pitch_peak_scale_kernel, dim3(grid_for(n, 512, 2)), dim3(512), (size_t)0, st, d_out, n, peak, n_tiles, target);
}

}  // namespace ds

using namespace ds;

extern "C" {

int ds_pitch_shift_workspace(const long long* lengths, const double* n_steps, int B, long long* bytes, long long* stage_offsets) {
  DS_REQUIRE(bytes, "ds_pitch_shift_workspace: bytes must be non-null");
  PitchPlan p;
  int rc = plan_pitch(lengths, n_steps, B, "ds_pitch_shift_workspace", p);
  if (rc) return rc;
  *bytes = (long long)p.ws.bytes;
  if (stage_offsets) {
    stage_offsets[0] = (long long)p.off_D;
    stage_offsets[1] = (long long)p.off_S;
    stage_offsets[2] = (long long)p.off_frames;
    stage_offsets[3] = (long long)p.off_ys;
  }
  return DS_OK;
}

int ds_pitch_shift(const float* d_in, float* d_out, const long long* lengths, const double* n_steps, int B, void* d_ws, long long ws_bytes,
                   void* stream) {
  DS_REQUIRE(d_in && d_out && d_ws, "ds_pitch_shift: d_in, d_out and d_ws must be non-null");
  PitchPlan p;
  int rc = plan_pitch(lengths, n_steps, B, "ds_pitch_shift", p);
  if (rc) return rc;
  DS_REQUIRE(ws_bytes >= (long long)p.ws.bytes, "ds_pitch_shift: workspace of %lld bytes, %zu needed", ws_bytes, p.ws.bytes);
  float2 *tw512, *tw1024, *tw2048;
  rc = get_twiddles((cudaStream_t)stream, &tw512, &tw1024, &tw2048);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)d_ws;
  const size_t n1 = (size_t)B + 1;
  const long long *loff = (const long long*)(ws + p.off_idx), *fin = loff + n1, *fout = fin + n1, *yoff = fout + n1, *tcap = yoff + n1,
                  *nval = tcap + B;
  const double* rate = (const double*)(ws + p.off_rate);
  float2* D = (float2*)(ws + p.off_D);
  float2* S = (float2*)(ws + p.off_S);
  float* frames = (float*)(ws + p.off_frames);
  float* ys = (float*)(ws + p.off_ys);
  DS_CHECK_CUDA(p.ws.upload(ws, st));
  const size_t smem = FR * XS_PITCH * sizeof(float2);
  DS_CHECK_CUDA(cudaFuncSetAttribute(pitch_stft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(cudaFuncSetAttribute(pitch_istft_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  DS_CHECK_CUDA(launch_pdl(pitch_stft_kernel, dim3((unsigned)((p.n_in_frames + FR - 1) / FR)), dim3(256), smem, st, d_in, loff, fin, B, D,
                           (const float2*)tw1024, (const float2*)tw2048));
  DS_CHECK_CUDA(launch_pdl(pitch_vocoder_kernel, dim3((unsigned)(((long long)B * NBIN + 255) / 256)), dim3(256), (size_t)0, st,
                           (const float2*)D, S, fin, fout, rate, B));
  DS_CHECK_CUDA(launch_pdl(pitch_istft_frames_kernel, dim3((unsigned)((p.n_out_frames + FR - 1) / FR)), dim3(256), smem, st,
                           (const float2*)S, frames, p.n_out_frames, (const float2*)tw1024, (const float2*)tw2048));
  DS_CHECK_CUDA(launch_pdl(pitch_ola_kernel, dim3(grid_for(p.n_ys, 256, 32)), dim3(256), (size_t)0, st, (const float*)frames, ys, fout,
                           yoff, tcap, B));
  DS_CHECK_CUDA(launch_pdl(pitch_resample_kernel, dim3(grid_for(p.n_samples, 256, 32)), dim3(256), (size_t)0, st, (const float*)ys, d_out,
                           loff, yoff, nval, rate, B, (float)(1.0 / bessel_i0(RS_BETA))));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_mix_track_workspace(const long long* lengths, const long long* onsets, int K, long long track_len, long long* bytes) {
  DS_REQUIRE(bytes, "ds_mix_track_workspace: bytes must be non-null");
  return mix_workspace(lengths, onsets, std::vector<long long>(K > 0 ? K : 0).data(), nullptr, K, 0.f, track_len, bytes,
                       "ds_mix_track_workspace");
}

int ds_mix_track(const float* d_src, const long long* src_off, const long long* lengths, const long long* onsets, const float* gains, int K,
                 float* d_track, long long track_len, void* d_ws, long long ws_bytes, void* stream) {
  DS_REQUIRE(d_src && d_track && d_ws && src_off && gains, "ds_mix_track: d_src, d_track, d_ws, src_off and gains must be non-null");
  return mix(d_src, src_off, lengths, onsets, gains, nullptr, std::vector<long long>(K > 0 ? K : 0).data(), K, 0.f, d_track, track_len,
             d_ws, ws_bytes, stream, "ds_mix_track");
}

int ds_mix_arrangement_workspace(const long long* lengths, const long long* onsets, const long long* fade_out, int K, float target_peak,
                                 long long track_len, long long* bytes) {
  DS_REQUIRE(bytes && fade_out, "ds_mix_arrangement_workspace: bytes and fade_out must be non-null");
  return mix_workspace(lengths, onsets, fade_out, nullptr, K, target_peak, track_len, bytes, "ds_mix_arrangement_workspace");
}

int ds_mix_arrangement(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets,
                       const float* gains, const long long* fade_out, int K, float target_peak, float* d_track, long long track_len,
                       void* d_ws, long long ws_bytes, void* stream) {
  DS_REQUIRE(d_src && d_track && d_ws && src_offsets && gains && fade_out,
             "ds_mix_arrangement: d_src, d_track, d_ws, src_offsets, gains and fade_out must be non-null");
  return mix(d_src, src_offsets, lengths, onsets, gains, nullptr, fade_out, K, target_peak, d_track, track_len, d_ws, ws_bytes, stream,
             "ds_mix_arrangement");
}

int ds_mix_stereo_workspace(const long long* lengths, const long long* onsets, const long long* fade_out, const float* pans, int K,
                            float target_peak, long long track_len, long long* bytes) {
  DS_REQUIRE(bytes && fade_out && pans, "ds_mix_stereo_workspace: bytes, fade_out and pans must be non-null");
  return mix_workspace(lengths, onsets, fade_out, pans, K, target_peak, track_len, bytes, "ds_mix_stereo_workspace");
}

int ds_mix_stereo(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets, const float* gains,
                  const float* pans, const long long* fade_out, int K, float target_peak, float* d_out, long long track_len, void* d_ws,
                  long long ws_bytes, void* stream) {
  DS_REQUIRE(d_src && d_out && d_ws && src_offsets && gains && pans && fade_out,
             "ds_mix_stereo: d_src, d_out, d_ws, src_offsets, gains, pans and fade_out must be non-null");
  return mix(d_src, src_offsets, lengths, onsets, gains, pans, fade_out, K, target_peak, d_out, track_len, d_ws, ws_bytes, stream,
             "ds_mix_stereo");
}

}  // extern "C"
