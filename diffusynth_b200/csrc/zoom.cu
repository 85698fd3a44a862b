// Mask zoom for inpainting with text (inpaint_with_text.py: the spectrogram mask is shrunk to the latent grid):
//   scipy.ndimage.zoom(a, (h / H, w / W))  with scipy's defaults order=3, mode='constant', prefilter=True, grid_mode=False,
// for B 2-D fp32 arrays packed back to back (item k: H_k x W_k in, h_k x w_k out).  The operation is separable, so each axis is
// prefiltered and interpolated in turn, in float64 as scipy does:
//   prefilter: cubic B-spline, pole z = sqrt(3) - 2, gain (1 - z)(1 - 1/z), mirror boundary, scipy's exact causal init
//     c0 = (x0 + z^(n-1) x_{n-1} + sum_{i=1}^{n-2} z^i (x_i + z^(n-1) x_{n-1-i})) / (1 - z^(2n-2)), c_i += z c_{i-1},
//     anticausal init c_{n-1} = z / (z^2 - 1) (z c_{n-2} + c_{n-1}), c_i = z (c_{i+1} - c_i); a line of length 1 is unchanged;
//   interpolation: output o samples x = o * ((n - 1) / (out - 1)) (0 when out = 1) as the cubic-B-spline-weighted sum of the
//     coefficients floor(x) - 1 .. floor(x) + 2, mirrored with period 2n - 2 (grid_mode=False keeps x in [0, n - 1], so the
//     constant is never read).
// Pass 1 walks one column of one item per thread (neighbouring threads read neighbouring columns) and writes the h_k x W_k
// intermediate; pass 2 walks one output row per thread.  Every output sums in a fixed order, without atomics: an item's result
// does not depend on its batch.  Per-item descriptors and prefix offsets are uploaded once: 2 launches and 1 copy whatever B.
#include "common.cuh"
#include <vector>
#include "../../include/diffusynth_b200.h"

namespace ds {
namespace {

constexpr int THREADS = 64;                       // small blocks: the per-thread walks are latency-bound, so spread them over the SMs

struct ZmItem {
  long long in_off, out_off, mid_off;              // element offsets: input and its coefficients (H x W), output (h x w), intermediate (h x W)
  long long H, W, h, w;
};

constexpr int CH = 8;                             // values a thread loads before it uses them: the walks are serial, the loads need not be

__device__ __forceinline__ double pole() { return sqrt(3.0) - 2.0; }
__device__ __forceinline__ double gain() { return (1.0 - pole()) * (1.0 - 1.0 / pole()); }

// Cubic B-spline coefficients c[0], c[s], ..., c[(n-1) s] (n >= 2) of the line x(0), ..., x(n-1) (gain applied by x), in scipy's
// order of operations.  x may read c itself (in place): every x(i) is read before c[i s] is written.
template <class X>
__device__ __forceinline__ void prefilter(X x, double* c, long long n, long long s) {
  const double z = pole();
  const double zn1 = pow(z, (double)(n - 1));
  double c0 = x(0) + zn1 * x(n - 1);
  double zi = z;
#pragma unroll 4
  for (long long i = 1; i < n - 1; ++i) {
    c0 += zi * (x(i) + zn1 * x(n - 1 - i));
    zi *= z;
  }
  double prev = c0 / (1.0 - zn1 * zn1);
  c[0] = prev;
  double v[CH];
  long long i = 1;
  for (; i + CH <= n; i += CH) {                   // causal: c_i = x_i + z c_{i-1}
#pragma unroll
    for (int j = 0; j < CH; ++j) v[j] = x(i + j);
#pragma unroll
    for (int j = 0; j < CH; ++j) { prev = v[j] + z * prev; c[(i + j) * s] = prev; }
  }
  for (; i < n; ++i) { prev = x(i) + z * prev; c[i * s] = prev; }
  double next = z / (z * z - 1.0) * (z * c[(n - 2) * s] + prev);
  c[(n - 1) * s] = next;
  i = n - 2;
  for (; i + 1 >= CH; i -= CH) {                   // anticausal: c_i = z (c_{i+1} - c_i)
#pragma unroll
    for (int j = 0; j < CH; ++j) v[j] = c[(i - j) * s];
#pragma unroll
    for (int j = 0; j < CH; ++j) { next = z * (next - v[j]); c[(i - j) * s] = next; }
  }
  for (; i >= 0; --i) { next = z * (next - c[i * s]); c[i * s] = next; }
}

__device__ __forceinline__ long long mirror(long long k, long long n) {
  if (n == 1) return 0;
  const long long p = 2 * n - 2;
  k = (k < 0 ? -k : k) % p;
  return k >= n ? p - k : k;
}

// Output o of a line of n coefficients c[0], c[s], ... zoomed to `out` samples.
__device__ __forceinline__ double interpolate(const double* c, long long n, long long s, long long o, long long out) {
  const double step = out > 1 ? (double)(n - 1) / (double)(out - 1) : 0.0;
  const double x = (double)o * step, f = floor(x), t = x - f, u = 1.0 - t;
  const double w0 = u * u * u / 6.0, w1 = (3.0 * t * t * (t - 2.0) + 4.0) / 6.0;
  const double w2 = (3.0 * u * u * (u - 2.0) + 4.0) / 6.0, w3 = t * t * t / 6.0;
  const long long b = (long long)f;
  return w0 * c[mirror(b - 1, n) * s] + w1 * c[mirror(b, n) * s] + w2 * c[mirror(b + 1, n) * s] + w3 * c[mirror(b + 2, n) * s];
}

// All `out` samples of the line, CH at a time (loads of a chunk before its stores); store(o, value).
template <class St>
__device__ __forceinline__ void interpolate_line(const double* c, long long n, long long s, long long out, St store) {
  for (long long o0 = 0; o0 < out; o0 += CH) {
    double r[CH];
#pragma unroll
    for (int j = 0; j < CH; ++j) r[j] = o0 + j < out ? interpolate(c, n, s, o0 + j, out) : 0.0;
#pragma unroll
    for (int j = 0; j < CH; ++j)
      if (o0 + j < out) store(o0 + j, r[j]);
  }
}

// ---- pass 1: one thread per (item, column): prefilter the H_k values, interpolate h_k of them -------------------------------
__global__ void __launch_bounds__(THREADS)
zoom_cols_kernel(const float* __restrict__ in, const ZmItem* __restrict__ items, const long long* __restrict__ colpre, int B,
                 double* __restrict__ coef, double* __restrict__ mid) {
  pdl_enter();
  const long long total = __ldg(colpre + B);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int k = find_item(colpre, B, g);
    const ZmItem it = items[k];
    const long long col = g - __ldg(colpre + k), W = it.W;
    const float* src = in + it.in_off + col;
    double* c = coef + it.in_off + col;
    if (it.H == 1) c[0] = (double)__ldg(src);
    else prefilter([=](long long i) { return (double)__ldg(src + i * W) * gain(); }, c, it.H, W);
    double* dst = mid + it.mid_off + col;
    interpolate_line(c, it.H, W, it.h, [=](long long o, double v) { dst[o * W] = v; });
  }
}

// ---- pass 2: one thread per (item, output row): prefilter the W_k values of its intermediate row in place, interpolate w_k -----
__global__ void __launch_bounds__(THREADS)
zoom_rows_kernel(const ZmItem* __restrict__ items, const long long* __restrict__ rowpre, int B, double* __restrict__ mid,
                 float* __restrict__ out) {
  pdl_enter();
  const long long total = __ldg(rowpre + B);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int k = find_item(rowpre, B, g);
    const ZmItem it = items[k];
    const long long r = g - __ldg(rowpre + k);
    double* c = mid + it.mid_off + r * it.W;
    if (it.W > 1) prefilter([=](long long i) { return c[i] * gain(); }, c, it.W, 1);
    float* dst = out + it.out_off + r * it.w;
    interpolate_line(c, it.W, 1, it.w, [=](long long o, double v) { dst[o] = (float)v; });
  }
}

struct ZoomPlan {
  std::vector<ZmItem> items;
  std::vector<long long> colpre, rowpre;
  Workspace ws;
  size_t off_items = 0, off_colpre = 0, off_rowpre = 0, off_coef = 0, off_mid = 0;
};

int plan_zoom(const long long* in_shapes, const long long* out_shapes, int B, const char* who, ZoomPlan& p) {
  DS_REQUIRE(in_shapes && out_shapes && B > 0, "%s: in_shapes and out_shapes must be non-null and B > 0 (B = %d)", who, B);
  for (int k = 0; k < B; ++k) {
    const long long H = in_shapes[2 * k], W = in_shapes[2 * k + 1], h = out_shapes[2 * k], w = out_shapes[2 * k + 1];
    DS_REQUIRE(H > 0 && W > 0 && h > 0 && w > 0 && H <= DS_MASK_ZOOM_MAX_DIM && W <= DS_MASK_ZOOM_MAX_DIM && h <= DS_MASK_ZOOM_MAX_DIM &&
                   w <= DS_MASK_ZOOM_MAX_DIM,
               "%s: item %d is %lld x %lld -> %lld x %lld (every dimension must be in 1..%lld)", who, k, H, W, h, w,
               (long long)DS_MASK_ZOOM_MAX_DIM);
  }
  p.items.assign(B, ZmItem{});
  p.colpre.assign(B + 1, 0);
  p.rowpre.assign(B + 1, 0);
  long long in_off = 0, out_off = 0, mid_off = 0;
  for (int k = 0; k < B; ++k) {
    ZmItem& it = p.items[k];
    it.H = in_shapes[2 * k];
    it.W = in_shapes[2 * k + 1];
    it.h = out_shapes[2 * k];
    it.w = out_shapes[2 * k + 1];
    it.in_off = in_off;
    it.out_off = out_off;
    it.mid_off = mid_off;
    in_off += it.H * it.W;
    out_off += it.h * it.w;
    mid_off += it.h * it.W;
    p.colpre[k + 1] = p.colpre[k] + it.W;
    p.rowpre[k + 1] = p.rowpre[k] + it.h;
  }
  p.off_items = p.ws.stage(p.items.data(), p.items.size());
  p.off_colpre = p.ws.stage(p.colpre.data(), p.colpre.size());
  p.off_rowpre = p.ws.stage(p.rowpre.data(), p.rowpre.size());
  p.off_coef = p.ws.reserve((size_t)in_off * sizeof(double));
  p.off_mid = p.ws.reserve((size_t)mid_off * sizeof(double));
  return DS_OK;
}

}  // namespace
}  // namespace ds

using namespace ds;

extern "C" {

int ds_mask_zoom_workspace(const long long* in_shapes, const long long* out_shapes, int B, long long* bytes) {
  DS_REQUIRE(bytes, "ds_mask_zoom_workspace: bytes must be non-null");
  ZoomPlan p;
  int rc = plan_zoom(in_shapes, out_shapes, B, "ds_mask_zoom_workspace", p);
  if (rc) return rc;
  *bytes = (long long)p.ws.bytes;
  return DS_OK;
}

int ds_mask_zoom(const float* d_in, float* d_out, const long long* in_shapes, const long long* out_shapes, int B, void* d_ws,
                 long long ws_bytes, void* stream) {
  DS_REQUIRE(d_in && d_out && d_ws, "ds_mask_zoom: d_in, d_out and d_ws must be non-null");
  ZoomPlan p;
  int rc = plan_zoom(in_shapes, out_shapes, B, "ds_mask_zoom", p);
  if (rc) return rc;
  DS_REQUIRE(ws_bytes >= (long long)p.ws.bytes, "ds_mask_zoom: workspace of %lld bytes, %zu needed", ws_bytes, p.ws.bytes);
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)d_ws;
  const ZmItem* items = (const ZmItem*)(ws + p.off_items);
  double* coef = (double*)(ws + p.off_coef);
  double* mid = (double*)(ws + p.off_mid);
  DS_CHECK_CUDA(p.ws.upload(ws, st));
  DS_CHECK_CUDA(launch_pdl(zoom_cols_kernel, dim3(grid_for(p.colpre[B], THREADS, 16)), dim3(THREADS), (size_t)0, st, d_in, items,
                           (const long long*)(ws + p.off_colpre), B, coef, mid));
  DS_CHECK_CUDA(launch_pdl(zoom_rows_kernel, dim3(grid_for(p.rowpre[B], THREADS, 16)), dim3(THREADS), (size_t)0, st, items,
                           (const long long*)(ws + p.off_rowpre), B, mid, d_out));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
