// Timbre morph rows (DiffSynthSampler.interpolate's generate_linear_noise, model/DiffSynthSampler.py:224-269, batched): P
// sequences x N frames of initial noise and condition, row p*N + k = frame k of sequence p, a_k = k / (N - 1).
//   linear (reference :170-174): row = fl(fl(a e1) + fl((1 - a) e0)), with a and 1 - a evaluated in double and rounded to fp32
//     as torch rounds a Python scalar, and no FMA contraction: bit-identical to generate_linear_noise on the device;
//   slerp: theta = acos(clamp(<e0,e1> / (|e0| |e1|), -1, 1)) from a float64 reduction in a fixed order, then
//     row = fl(w0 e0 + w1 e1), w0 = sin((1 - a) theta) / sin theta, w1 = sin(a theta) / sin theta, weights and products in float64;
//     a sequence with sin theta < 1e-6 (identical or antipodal endpoints) or a zero endpoint takes the linear rows.
// Conditions always take the linear expression, except that an element equal in both endpoints is copied.  The reduction runs per sequence over fixed CHUNK-element blocks, each summing in
// a fixed order, and the row kernel adds the chunk partials in chunk order: a sequence's rows do not depend on P.
#include "common.cuh"
#include "../../include/diffusynth_b200.h"

namespace ds {
namespace {

constexpr int THREADS = 256;
constexpr long long CHUNK = 8192;                 // endpoint elements per partial (2048 float4, 8 per thread)
constexpr int ROW_VEC = 4;                        // float4 of noise per thread of the row kernel

struct Partial { double dot, n0, n1; };

__global__ void __launch_bounds__(THREADS)
morph_partials_kernel(const float4* __restrict__ e0, const float4* __restrict__ e1, long long nq, int nchunks, Partial* __restrict__ part) {
  pdl_enter();
  const long long p = blockIdx.x / nchunks;
  const int c = (int)(blockIdx.x - p * nchunks);
  const long long base = (long long)p * nq, lo = c * (CHUNK / 4), hi = min(lo + CHUNK / 4, nq);
  double d = 0.0, s0 = 0.0, s1 = 0.0;
  for (long long i = lo + threadIdx.x; i < hi; i += THREADS) {
    const float4 a = __ldg(e0 + base + i), b = __ldg(e1 + base + i);
    const double ax[4] = {a.x, a.y, a.z, a.w}, bx[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      d = __dadd_rn(d, __dmul_rn(ax[j], bx[j]));
      s0 = __dadd_rn(s0, __dmul_rn(ax[j], ax[j]));
      s1 = __dadd_rn(s1, __dmul_rn(bx[j], bx[j]));
    }
  }
  d = warp_sum(d);
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  __shared__ double sh[3][THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][warp] = d; sh[1][warp] = s0; sh[2][warp] = s1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    Partial r{0.0, 0.0, 0.0};
    for (int w = 0; w < THREADS / 32; ++w) { r.dot += sh[0][w]; r.n0 += sh[1][w]; r.n1 += sh[2][w]; }
    part[blockIdx.x] = r;
  }
}

// One block row of the grid = one output row (p, k); blockIdx.y walks its columns: noise as float4, conditions as scalars.
__global__ void __launch_bounds__(THREADS)
morph_rows_kernel(const float4* __restrict__ e0, const float4* __restrict__ e1, const float* __restrict__ c0, const float* __restrict__ c1,
                  int N, long long nq, long long L, const Partial* __restrict__ part, int nchunks, float4* __restrict__ noise,
                  float* __restrict__ cond) {
  pdl_enter();
  const long long row = blockIdx.x;
  const long long p = row / N;
  const int k = (int)(row - p * N);
  const double a = (double)k / (double)(N - 1);
  const float af = (float)a, bf = (float)(1.0 - a);
  __shared__ double w_sh[2];
  __shared__ int slerp_sh;
  if (threadIdx.x == 0) {
    int use = 0;
    if (part != nullptr) {
      double d = 0.0, s0 = 0.0, s1 = 0.0;
      for (int c = 0; c < nchunks; ++c) {
        const Partial q = part[p * nchunks + c];
        d += q.dot; s0 += q.n0; s1 += q.n1;
      }
      if (s0 > 0.0 && s1 > 0.0) {
        const double cs = fmin(fmax(d / (sqrt(s0) * sqrt(s1)), -1.0), 1.0);
        const double th = acos(cs), st = sin(th);
        if (st >= 1e-6) {
          w_sh[0] = sin((1.0 - a) * th) / st;
          w_sh[1] = sin(a * th) / st;
          use = 1;
        }
      }
    }
    slerp_sh = use;
  }
  __syncthreads();
  const bool slerp = slerp_sh != 0;
  const double w0 = slerp ? w_sh[0] : 0.0, w1 = slerp ? w_sh[1] : 0.0;
  const long long src = p * nq, dst = row * nq;
  const long long g0 = (long long)blockIdx.y * (THREADS * ROW_VEC) + threadIdx.x;
#pragma unroll
  for (int j = 0; j < ROW_VEC; ++j) {
    const long long i = g0 + (long long)j * THREADS;
    if (i < nq) {
      const float4 x = __ldg(e0 + src + i), y = __ldg(e1 + src + i);
      float4 r;
      if (slerp) {
        r.x = (float)__dadd_rn(__dmul_rn(w0, (double)x.x), __dmul_rn(w1, (double)y.x));
        r.y = (float)__dadd_rn(__dmul_rn(w0, (double)x.y), __dmul_rn(w1, (double)y.y));
        r.z = (float)__dadd_rn(__dmul_rn(w0, (double)x.z), __dmul_rn(w1, (double)y.z));
        r.w = (float)__dadd_rn(__dmul_rn(w0, (double)x.w), __dmul_rn(w1, (double)y.w));
      } else {
        r.x = __fadd_rn(__fmul_rn(af, y.x), __fmul_rn(bf, x.x));
        r.y = __fadd_rn(__fmul_rn(af, y.y), __fmul_rn(bf, x.y));
        r.z = __fadd_rn(__fmul_rn(af, y.z), __fmul_rn(bf, x.z));
        r.w = __fadd_rn(__fmul_rn(af, y.w), __fmul_rn(bf, x.w));
      }
      noise[dst + i] = r;
    }
    if (i < L) {
      // an element the two conditions share is kept as it is: fl(a c) + fl((1 - a) c) may miss c by an ulp, and a morph under
      // one prompt must sample under exactly that prompt (as interpolate does)
      const float x = __ldg(c0 + p * L + i), y = __ldg(c1 + p * L + i);
      cond[row * L + i] = x == y ? x : __fadd_rn(__fmul_rn(af, y), __fmul_rn(bf, x));
    }
  }
}

long long num_chunks(long long n) { return (n + CHUNK - 1) / CHUNK; }

long long row_blocks(long long n, long long L) {
  const long long cols = n / 4 > L ? n / 4 : L;
  return (cols + THREADS * ROW_VEC - 1) / (THREADS * ROW_VEC);
}

int check_args(int P, int N, long long n, long long L, int path, const char* who) {
  DS_REQUIRE(P > 0 && N >= 2, "%s: P must be > 0 and N >= 2 (P = %d, N = %d)", who, P, N);
  DS_REQUIRE(n > 0 && n % 4 == 0, "%s: n must be a positive multiple of 4 (n = %lld)", who, n);
  DS_REQUIRE(L > 0, "%s: L must be > 0 (L = %lld)", who, L);
  DS_REQUIRE(path == DS_MORPH_LINEAR || path == DS_MORPH_SLERP, "%s: unknown path %d (DS_MORPH_LINEAR = 0, DS_MORPH_SLERP = 1)", who,
             path);
  long long rows = 0, elems = 0;
  DS_REQUIRE(!__builtin_mul_overflow((long long)P, (long long)N, &rows) && !__builtin_mul_overflow(rows, n > L ? n : L, &elems) &&
                 !__builtin_mul_overflow(elems, (long long)sizeof(float), &elems),
             "%s: P * N * max(n, L) = %d * %d * %lld overflows", who, P, N, n > L ? n : L);
  // launch geometry: one block row per output row, one partial block per (sequence, chunk), up to 65535 column blocks per row
  DS_REQUIRE(rows <= 0x7fffffffLL && (long long)P * num_chunks(n) <= 0x7fffffffLL && row_blocks(n, L) <= 65535,
             "%s: P = %d, N = %d, n = %lld, L = %lld exceed the launch geometry (P * N < 2^31, max(n / 4, L) <= %lld)", who, P, N, n, L,
             65535LL * THREADS * ROW_VEC);
  return DS_OK;
}

long long workspace_bytes(int P, long long n, int path) {
  return path == DS_MORPH_SLERP ? (long long)P * num_chunks(n) * (long long)sizeof(Partial) : 0;
}

}  // namespace
}  // namespace ds

using namespace ds;

extern "C" {

int ds_morph_rows_workspace(int P, int N, long long n, long long L, int path, long long* bytes) {
  DS_REQUIRE(bytes, "ds_morph_rows_workspace: bytes must be non-null");
  int rc = check_args(P, N, n, L, path, "ds_morph_rows_workspace");
  if (rc) return rc;
  *bytes = workspace_bytes(P, n, path);
  return DS_OK;
}

int ds_morph_rows(const float* d_e0, const float* d_e1, const float* d_c0, const float* d_c1, int P, int N, long long n, long long L,
                  int path, float* d_noise, float* d_cond, void* d_ws, long long ws_bytes, void* stream) {
  DS_REQUIRE(d_e0 && d_e1 && d_c0 && d_c1 && d_noise && d_cond, "ds_morph_rows: endpoint and output pointers must be non-null");
  int rc = check_args(P, N, n, L, path, "ds_morph_rows");
  if (rc) return rc;
  const long long need = workspace_bytes(P, n, path);
  DS_REQUIRE(need == 0 || d_ws, "ds_morph_rows: d_ws must be non-null for the slerp path");
  DS_REQUIRE(ws_bytes >= need, "ds_morph_rows: workspace of %lld bytes, %lld needed", ws_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const long long nq = n / 4;
  const int nchunks = (int)num_chunks(n);
  Partial* part = nullptr;
  if (path == DS_MORPH_SLERP) {
    part = (Partial*)d_ws;
    DS_CHECK_CUDA(launch_pdl(morph_partials_kernel, dim3((unsigned)((long long)P * nchunks)), dim3(THREADS), (size_t)0, st, (const float4*)d_e0,
                             (const float4*)d_e1, nq, nchunks, part));
  }
  DS_CHECK_CUDA(launch_pdl(morph_rows_kernel, dim3((unsigned)((long long)P * N), (unsigned)row_blocks(n, L)), dim3(THREADS), (size_t)0, st,
                           (const float4*)d_e0, (const float4*)d_e1, d_c0, d_c1, N, nq, L, (const Partial*)part, nchunks,
                           (float4*)d_noise, d_cond));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
