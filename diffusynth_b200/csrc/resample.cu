// Sample-rate conversion for uploaded audio (tools.adjust_audio_length, tools.py:126-151, as the timbre-modification upload handler
// calls it, sound2sound_with_text.py:75-82): optional peak normalisation, then
//   librosa.resample(x, orig_sr=o, target_sr=t, res_type="kaiser_best") -> fix_length(out_len)
// with the filter of pitch.cu's resampler (resampy's kaiser_best parameters; DESIGN.md section 8):
//   out[j] = sum_i xn[i] h(i - j*o/t),  h(d) = s*roll*sinc(s*roll*d) * I0(beta sqrt(1 - (s d / 64)^2)) / I0(beta),  |d| <= 64/s,
//   s = min(1, t/o), samples outside [0, L) zero, ceil(L * (t/o)) valid outputs (float64, librosa's length), zero past them.
// Sample rates are integers, so with g = gcd(o, t), up = t/g, down = o/g, output j sits at input (j*down) div up plus the phase
// (j*down) mod up / up, and the taps repeat over `up` phases.  A table [up][taps] of fp32 coefficients (evaluated in float64 on the
// device) turns each tap into one load and one FMA.  Pairs whose table or staged input window would be too large evaluate the same
// float64 coefficients per tap instead (the direct path): both paths sum the same fp32 products in ascending input order and give
// bit-identical results.  Equal rates copy, as librosa.resample returns its input.  Ragged batch: per-item descriptors and prefix
// offsets uploaded once, one launch per stage (table build, peak when normalising, resample) whatever the number of items.
#include "common.cuh"
#include <cmath>
#include <cstdlib>
#include <map>
#include <numeric>
#include <utility>
#include <vector>
#include "../../include/diffusynth_b200.h"

namespace ds {
namespace {

constexpr int THREADS = 256, WARPS = THREADS / 32;
constexpr long long TABLE_CAP = 1LL << 20;     // coefficients per (o, t) pair; larger tables take the direct path
constexpr int WIN_CAP = 24576;                 // staged input floats per CTA; a pair needing more takes the direct path
constexpr int WIN_TARGET = 16384;              // staged input floats a CTA aims for
constexpr int OUT_TARGET = 4096;               // outputs a table-path CTA aims for
constexpr int DIRECT_TILE = 1024, COPY_TILE = 4096, PEAK_TILE = 8192;
enum : long long { MODE_COPY = 0, MODE_TABLE = 1, MODE_DIRECT = 2 };

// Per-item descriptor (device copy is read-only).  Table path: a CTA owns outputs [tile * N * up, (tile + 1) * N * up).
struct RsItem {
  long long in_off, len, out_off, out_len, nval;   // packed offsets, input length, written length, valid outputs (librosa's)
  long long up, down, F, taps4;                    // F = floor(64 / s): taps m in [-F, F + 1]; taps4 = 2F + 2 rounded up to 4
  long long mode, tab_off, N, tile_out;            // tab_off: first coefficient of the item's table (table path)
  double ratio;                                    // t / o as numpy evaluates it
};
struct RsPair {
  long long up, down, F, taps4;
  double ratio;
};

// h(m - p/up) in float64, rounded once to fp32; zero outside the filter's support |m - p/up| <= 64/s, which is decided in integers
// (|m*up - p| <= 64*max(up, down)) so that the taps exactly at the edge count.  Shared by the table build and the direct path, so
// both paths multiply by the same fp32 coefficients.
__device__ __forceinline__ float rs_tap(long long m, long long p, long long up, long long down, double ratio, double inv_i0) {
  const long long reach = m * up - p;
  if ((reach < 0 ? -reach : reach) > RS_ZEROS * (up > down ? up : down)) return 0.f;
  const double sc = ratio < 1.0 ? ratio : 1.0;
  const double d = (double)m - (double)p / (double)up;
  const double u = d * (sc / RS_ZEROS);
  const double cut = sc * RS_ROLLOFF, z = cut * d;
  const double sinc = z == 0.0 ? 1.0 : sinpi(z) / (kPi * z);
  return (float)(cut * sinc * cyl_bessel_i0(RS_BETA * sqrt(fmax(0.0, 1.0 - u * u))) * inv_i0);
}

// peak normaliser of item k: max(max|x|, 1e-12), NaN propagated like torch's amax / clamp_min
__device__ __forceinline__ float rs_peak(const unsigned* __restrict__ peak, int k) {
  const float v = __uint_as_float(peak[k]);
  return v < 1e-12f ? 1e-12f : v;
}

// ---- coefficient tables of every distinct table-path pair, and the zeroing of the per-item peaks -----------------------------
__global__ void __launch_bounds__(THREADS)
resample_table_kernel(const RsPair* __restrict__ pairs, const long long* __restrict__ poff, int P, float* __restrict__ tab,
                      unsigned* __restrict__ peak, int B) {
  pdl_enter();
  const long long g0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
  for (long long g = g0; g < B; g += stride) peak[g] = 0u;
  if (P == 0) return;
  const double inv_i0 = 1.0 / cyl_bessel_i0(RS_BETA);
  const long long total = __ldg(poff + P);
  for (long long g = g0; g < total; g += stride) {
    const int q = find_item(poff, P, g);
    const RsPair pr = pairs[q];
    const long long e = g - __ldg(poff + q), p = e / pr.taps4, c = e - p * pr.taps4;
    tab[g] = c < 2 * pr.F + 2 ? rs_tap(c - pr.F, p, pr.up, pr.down, pr.ratio, inv_i0) : 0.f;
  }
}

// ---- per-item max |x|: one block per PEAK_TILE samples, an integer atomicMax on the bits of the non-negative block maximum -----
__global__ void __launch_bounds__(THREADS)
resample_peak_kernel(const float* __restrict__ x, const RsItem* __restrict__ items, const long long* __restrict__ ptile, int B,
                     unsigned* __restrict__ peak) {
  pdl_enter();
  __shared__ unsigned red[WARPS];
  const int k = find_item(ptile, B, blockIdx.x);
  const RsItem& it = items[k];
  const long long lo = (blockIdx.x - __ldg(ptile + k)) * (long long)PEAK_TILE;
  const long long hi = lo + PEAK_TILE < it.len ? lo + PEAK_TILE : it.len;
  const float* src = x + it.in_off;
  unsigned m = 0u;                                           // bits of |x| order like the values (NaN above +inf)
  for (long long i = lo + threadIdx.x; i < hi; i += THREADS) m = max(m, __float_as_uint(fabsf(__ldg(src + i))));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < WARPS; ++w) m = max(m, red[w]);
    atomicMax(peak + k, m);
  }
}

// staged window index -> shared-memory slot.  With an even `down`, lanes that read `down` samples apart would share banks; one
// pad slot per 32 samples spreads them.
template <bool SKEW>
__device__ __forceinline__ int wslot(int w) { return SKEW ? w + (w >> 5) : w; }

// Table path of one CTA: output j = J0 + q*up + r (q < N, r < up) has phase p = (r*down) mod up and reads window samples
// q*down + (r*down) div up + c, c = 0 .. taps4-1 (tap m = c - F).  A warp takes 32 consecutive q of one r, so the coefficient row
// is warp-uniform and read 4 taps at a time.
template <bool SKEW>
__device__ __forceinline__ void table_tile(const float* __restrict__ xs, const float* __restrict__ tab, const RsItem& it, long long J0,
                                           float* __restrict__ out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int qchunks = (int)(it.N / 32), nch = (int)it.up * qchunks, taps4 = (int)it.taps4;
  for (int ch = warp; ch < nch; ch += WARPS) {
    const int r = ch / qchunks, q = (ch - r * qchunks) * 32 + lane;
    const long long j = J0 + (long long)q * it.up + r;
    if (j >= it.out_len) continue;
    float acc = 0.f;
    if (j < it.nval) {
      const long long rd = (long long)r * it.down;
      const long long p = rd % it.up;
      const int w0 = q * (int)it.down + (int)(rd / it.up);
      const float4* row = reinterpret_cast<const float4*>(tab + p * it.taps4);
#pragma unroll 2
      for (int c = 0; c < taps4; c += 4) {
        const float4 h = __ldg(row + (c >> 2));
        acc = fmaf(xs[wslot<SKEW>(w0 + c)], h.x, acc);
        acc = fmaf(xs[wslot<SKEW>(w0 + c + 1)], h.y, acc);
        acc = fmaf(xs[wslot<SKEW>(w0 + c + 2)], h.z, acc);
        acc = fmaf(xs[wslot<SKEW>(w0 + c + 3)], h.w, acc);
      }
    }
    out[j] = acc;
  }
}

// ---- resample + fix_length: one CTA per tile of one item's outputs ---------------------------------------------------------
__global__ void __launch_bounds__(THREADS)
resample_kernel(const float* __restrict__ x, float* __restrict__ y, const RsItem* __restrict__ items, const long long* __restrict__ tiles,
                int B, const float* __restrict__ tab, const unsigned* __restrict__ peak, int normalize) {
  pdl_enter();
  extern __shared__ float rs_xs[];
  const int k = find_item(tiles, B, blockIdx.x);
  const RsItem& it = items[k];
  const long long tile = blockIdx.x - __ldg(tiles + k), J0 = tile * it.tile_out;
  const float* src = x + it.in_off;
  float* out = y + it.out_off;
  const float pk = normalize ? rs_peak(peak, k) : 1.f;
  if (it.mode == MODE_TABLE && J0 < it.nval) {
    const long long W0 = tile * it.N * it.down - it.F;
    const int wlen = (int)((it.N - 1) * it.down + ((it.up - 1) * it.down) / it.up + it.taps4);
    const bool skew = (it.down & 1) == 0;
    for (int w = threadIdx.x; w < wlen; w += THREADS) {
      const long long i = W0 + w;
      float v = (i >= 0 && i < it.len) ? __ldg(src + i) : 0.f;
      if (normalize) v = v / pk;
      rs_xs[skew ? wslot<true>(w) : w] = v;
    }
    __syncthreads();
    if (skew) table_tile<true>(rs_xs, tab + it.tab_off, it, J0, out);
    else table_tile<false>(rs_xs, tab + it.tab_off, it, J0, out);
    return;
  }
  const double inv_i0 = it.mode == MODE_DIRECT ? 1.0 / cyl_bessel_i0(RS_BETA) : 0.0;
  for (int t = threadIdx.x; t < it.tile_out; t += THREADS) {
    const long long j = J0 + t;
    if (j >= it.out_len) break;
    float acc = 0.f;
    if (j < it.nval) {
      if (it.mode == MODE_COPY) {
        acc = __ldg(src + j);
        if (normalize) acc = acc / pk;
      } else if (it.mode == MODE_DIRECT) {                   // the table path's sum, coefficients evaluated per tap
        const long long jd = j * it.down, b = jd / it.up, p = jd - b * it.up;
        const long long c0 = it.F - b > 0 ? it.F - b : 0, c1 = it.len - 1 - b + it.F < 2 * it.F + 1 ? it.len - 1 - b + it.F : 2 * it.F + 1;
        for (long long c = c0; c <= c1; ++c) {
          float v = __ldg(src + b - it.F + c);
          if (normalize) v = v / pk;
          acc = fmaf(v, rs_tap(c - it.F, p, it.up, it.down, it.ratio, inv_i0), acc);
        }
      }
      // MODE_TABLE with J0 >= nval never reaches here with j < nval
    }
    out[j] = acc;
  }
}

struct ResamplePlan {
  std::vector<RsItem> items;
  std::vector<long long> tiles, ptiles, poff;            // prefix offsets: resample tiles, peak tiles, table coefficients
  std::vector<RsPair> pairs;
  Workspace ws;
  size_t off_items = 0, off_tiles = 0, off_ptiles = 0, off_pairs = 0, off_poff = 0, off_tab = 0, off_peak = 0, smem = 0;
};

int plan_resample(const long long* lengths, const long long* sr_in, const long long* sr_out, const long long* out_lengths, int B,
                  const char* who, ResamplePlan& p) {
  DS_REQUIRE(lengths && sr_in && sr_out && B > 0, "%s: lengths, sr_in and sr_out must be non-null and B > 0 (B = %d)", who, B);
  for (int k = 0; k < B; ++k) {
    DS_REQUIRE(lengths[k] > 0 && lengths[k] <= DS_RESAMPLE_MAX_LENGTH, "%s: item %d has length %lld (must be in 1..%lld)", who, k,
               lengths[k], (long long)DS_RESAMPLE_MAX_LENGTH);
    DS_REQUIRE(sr_in[k] > 0 && sr_in[k] <= DS_RESAMPLE_MAX_RATE && sr_out[k] > 0 && sr_out[k] <= DS_RESAMPLE_MAX_RATE,
               "%s: item %d has rates %lld -> %lld (must be in 1..%lld)", who, k, sr_in[k], sr_out[k], (long long)DS_RESAMPLE_MAX_RATE);
    if (out_lengths)
      DS_REQUIRE(out_lengths[k] > 0 && out_lengths[k] <= DS_RESAMPLE_MAX_LENGTH, "%s: item %d has output length %lld (must be in 1..%lld)",
                 who, k, out_lengths[k], (long long)DS_RESAMPLE_MAX_LENGTH);
  }
  const char* env = getenv("DS_RESAMPLE_DIRECT");             // A/B timing and tests: every resampled item takes the direct path
  const bool force_direct = env && atoi(env) != 0;
  p.items.assign(B, RsItem{});
  p.tiles.assign(B + 1, 0);
  p.ptiles.assign(B + 1, 0);
  p.pairs.clear();
  p.poff.assign(1, 0);
  std::map<std::pair<long long, long long>, long long> table_of;   // (o, t) -> first coefficient
  long long in_off = 0, out_off = 0;
  size_t smem_floats = 0;
  for (int k = 0; k < B; ++k) {
    RsItem& it = p.items[k];
    const long long o = sr_in[k], t = sr_out[k], L = lengths[k], g = std::gcd(o, t);
    it.in_off = in_off;
    it.len = L;
    it.out_off = out_off;
    it.ratio = (double)t / (double)o;
    it.nval = (long long)std::ceil((double)L * it.ratio);     // librosa.resample: int(np.ceil(n * float(target_sr) / orig_sr))
    it.out_len = out_lengths ? out_lengths[k] : it.nval;
    it.up = t / g;
    it.down = o / g;
    const double sc = it.ratio < 1.0 ? it.ratio : 1.0;
    it.F = (long long)std::floor(RS_ZEROS / sc);
    it.taps4 = (2 * it.F + 2 + 3) & ~3LL;
    if (o == t) {
      it.mode = MODE_COPY;
      it.nval = L;
      if (!out_lengths) it.out_len = L;
      it.tile_out = COPY_TILE;
    } else if (!force_direct && it.up * it.taps4 <= TABLE_CAP && 32 * it.down + it.taps4 + 1 <= WIN_CAP) {
      it.mode = MODE_TABLE;
      long long nq = OUT_TARGET / (32 * it.up);
      const long long qwin = (WIN_TARGET - it.taps4 - 1) / (32 * it.down);
      if (nq > qwin) nq = qwin;
      if (nq < 1) nq = 1;
      it.N = 32 * nq;
      it.tile_out = it.N * it.up;
      const long long wlen = (it.N - 1) * it.down + ((it.up - 1) * it.down) / it.up + it.taps4;
      const size_t need = (size_t)(wlen + wlen / 32 + 1);
      if (need > smem_floats) smem_floats = need;
      auto key = std::make_pair(o, t);
      auto f = table_of.find(key);
      if (f == table_of.end()) {
        f = table_of.emplace(key, p.poff.back()).first;
        p.pairs.push_back(RsPair{it.up, it.down, it.F, it.taps4, it.ratio});
        p.poff.push_back(p.poff.back() + it.up * it.taps4);
      }
      it.tab_off = f->second;
    } else {
      it.mode = MODE_DIRECT;
      it.tile_out = DIRECT_TILE;
    }
    in_off += L;
    out_off += it.out_len;
    p.tiles[k + 1] = p.tiles[k] + (it.out_len + it.tile_out - 1) / it.tile_out;
    p.ptiles[k + 1] = p.ptiles[k] + (L + PEAK_TILE - 1) / PEAK_TILE;
  }
  p.off_items = p.ws.stage(p.items.data(), p.items.size());
  p.off_tiles = p.ws.stage(p.tiles.data(), p.tiles.size());
  p.off_ptiles = p.ws.stage(p.ptiles.data(), p.ptiles.size());
  p.off_pairs = p.ws.stage(p.pairs.data(), p.pairs.size());
  p.off_poff = p.ws.stage(p.poff.data(), p.poff.size());
  p.off_tab = p.ws.reserve((size_t)p.poff.back() * sizeof(float));
  p.off_peak = p.ws.reserve((size_t)B * sizeof(unsigned));
  p.smem = smem_floats * sizeof(float);
  return DS_OK;
}

}  // namespace
}  // namespace ds

using namespace ds;

extern "C" {

int ds_resample_workspace(const long long* lengths, const long long* sr_in, const long long* sr_out, const long long* out_lengths, int B,
                          long long* bytes) {
  DS_REQUIRE(bytes, "ds_resample_workspace: bytes must be non-null");
  ResamplePlan p;
  int rc = plan_resample(lengths, sr_in, sr_out, out_lengths, B, "ds_resample_workspace", p);
  if (rc) return rc;
  *bytes = (long long)p.ws.bytes;
  return DS_OK;
}

int ds_resample(const float* d_in, float* d_out, const long long* lengths, const long long* sr_in, const long long* sr_out,
                const long long* out_lengths, int normalize_peak, int B, void* d_ws, long long ws_bytes, void* stream) {
  DS_REQUIRE(d_in && d_out && d_ws, "ds_resample: d_in, d_out and d_ws must be non-null");
  ResamplePlan p;
  int rc = plan_resample(lengths, sr_in, sr_out, out_lengths, B, "ds_resample", p);
  if (rc) return rc;
  DS_REQUIRE(ws_bytes >= (long long)p.ws.bytes, "ds_resample: workspace of %lld bytes, %zu needed", ws_bytes, p.ws.bytes);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)d_ws;
  const RsItem* items = (const RsItem*)(ws + p.off_items);
  const long long* tiles = (const long long*)(ws + p.off_tiles);
  const long long* ptiles = (const long long*)(ws + p.off_ptiles);
  float* tab = (float*)(ws + p.off_tab);
  unsigned* peak = (unsigned*)(ws + p.off_peak);
  DS_CHECK_CUDA(p.ws.upload(ws, st));
  const long long n_coef = p.poff.back();
  DS_CHECK_CUDA(launch_pdl(resample_table_kernel, dim3(grid_for(n_coef > B ? n_coef : B, THREADS, 32)), dim3(THREADS), (size_t)0, st,
                           (const RsPair*)(ws + p.off_pairs), (const long long*)(ws + p.off_poff), (int)p.pairs.size(), tab, peak, B));
  if (normalize_peak)
    DS_CHECK_CUDA(launch_pdl(resample_peak_kernel, dim3((unsigned)p.ptiles[B]), dim3(THREADS), (size_t)0, st, d_in, items, ptiles, B,
                             peak));
  DS_CHECK_CUDA(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  DS_CHECK_CUDA(launch_pdl(resample_kernel, dim3((unsigned)p.tiles[B]), dim3(THREADS), p.smem, st, d_in, d_out, items, tiles, B,
                           (const float*)tab, (const unsigned*)peak, normalize_peak ? 1 : 0));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
