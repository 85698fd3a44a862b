// Shared helpers for the diffusynth_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <vector>

namespace ds {

// ---- error plumbing (C-ABI returns int; message kept per host thread) ------------------------
enum : int { DS_OK = 0, DS_ERR_INVALID = -1, DS_ERR_CUDA = -2, DS_ERR_NCCL = -3, DS_ERR_UNSUPPORTED = -4 };
void set_error(const char* fmt, ...);
const char* get_error();

#define DS_CHECK_CUDA(expr)                                                               \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ds::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return ds::DS_ERR_CUDA;                                                             \
    }                                                                                     \
  } while (0)

#define DS_REQUIRE(cond, ...)                 \
  do {                                        \
    if (!(cond)) {                            \
      ds::set_error(__VA_ARGS__);             \
      return ds::DS_ERR_INVALID;              \
    }                                         \
  } while (0)

// SM count of the CURRENT device (cached per device: one process may drive several GPUs).
inline int num_sms() {
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  int n = cache[dev];
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    cache[dev] = n;      // (benign race: every thread computes the same value)
  }
  return n;
}

// Blocks of `block` threads for n work items: ceil(n / block), at most per_sm per SM (grid-stride kernels) and at least 1.
inline unsigned grid_for(long long n, int block, int per_sm) {
  long long b = (n + block - 1) / block;
  const long long cap = (long long)num_sms() * per_sm;
  if (b > cap) b = cap;
  return (unsigned)(b > 0 ? b : 1);
}

inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// ---- workspace of a ragged-batch entry point ------------------------------------------------------------------------------
// stage() places a host array after the previous one, at its type's alignment, in one block at the start of the workspace, and
// returns its byte offset; reserve(), called after the last stage(), places device-only scratch after that block.  The block and
// every scratch buffer start 256-byte aligned; `bytes` is the workspace size.  The arrays are read only by upload(), so they must
// stay alive and unchanged until then (a workspace query plans the same way and never uploads).  upload() gathers them into a
// pageable host block and copies it with one cudaMemcpyAsync.  From a pageable source the copy is staged before the call returns,
// so the block may be freed at once; for the same reason these uploads are never made under stream capture, where the copy would
// read the freed block at every replay.
struct Workspace {
  struct Array { size_t off; const void* src; size_t n; };
  std::vector<Array> arrays;
  size_t staged = 0, bytes = 0;

  template <typename T>
  size_t stage(const T* src, size_t count) {
    const size_t o = (staged + alignof(T) - 1) / alignof(T) * alignof(T);
    arrays.push_back({o, src, count * sizeof(T)});
    staged = o + count * sizeof(T);
    bytes = align256(staged);
    return o;
  }
  size_t reserve(size_t n) {
    const size_t o = bytes;
    bytes = align256(o + n);
    return o;
  }
  cudaError_t upload(void* ws, cudaStream_t stream) const {
    std::vector<uint8_t> host(staged, 0);
    for (const Array& a : arrays)
      if (a.n) memcpy(host.data() + a.off, a.src, a.n);
    return cudaMemcpyAsync(ws, host.data(), staged, cudaMemcpyHostToDevice, stream);
  }
};

// Peak normalisation (pitch.cu; the arrangement mixes and convolve.cu): reduces n_tiles max |x| partials on the device and scales
// d_out[0, n) in place by target / max, leaving an all-zero output zero.  One PDL launch, no host synchronisation.
cudaError_t launch_peak_scale(float* d_out, long long n, const float* peak, int n_tiles, float target, cudaStream_t st);

// resampy's kaiser_best filter (pitch.cu, resample.cu): 64 zero crossings per side, roll-off and Kaiser beta
constexpr double kPi = 3.14159265358979323846;
constexpr int RS_ZEROS = 64;
constexpr double RS_ROLLOFF = 0.9475937167399596, RS_BETA = 14.769656459379492;

// ---- programmatic dependent launch ------------------------------------------------------------------------------
// Every hot-path kernel is launched with cudaLaunchAttributeProgrammaticStreamSerialization: its blocks may be scheduled while
// the previous kernel of the stream is still draining, run their prologue (barrier init, tensor-memory allocation, weight
// tables), and block in griddepcontrol.wait until that kernel has completed and its writes are visible.  A kernel touches
// activations (reads OR writes) only after pdl_wait(); since every kernel waits, the ordering is transitive along the stream.
// DS_PDL=0 (read once) launches everything with plain stream serialisation (A/B timing).
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("DS_PDL"); return !e || atoi(e) != 0; }();
  return on;
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- device helpers ---------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() { pdl_launch_dependents(); pdl_wait(); }
// 16-bit storage / tensor-core operand type of activations and weights.
// Default: IEEE fp16 (tcgen05 kind::f16 with f16 inputs, fp32 accumulate).  bf16 activations cannot hold the
// classifier-free-guidance difference eps_c - eps_u (0.5% of |eps| at random init, below bf16 resolution), see
// DESIGN.md "Operand precision"; -DDS_OPERANDS_BF16 builds the bf16 variant for comparison.
#ifdef DS_OPERANDS_BF16
typedef __nv_bfloat16 act_t;
static constexpr int kOperandIsFp16 = 0;
__device__ __forceinline__ float lo16(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float hi16(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float act2f(act_t v) { return __bfloat162float(v); }
__device__ __forceinline__ act_t f2act(float v) { return __float2bfloat16_rn(v); }
#else
typedef __half act_t;
static constexpr int kOperandIsFp16 = 1;
__device__ __forceinline__ float lo16(uint32_t v) { return __half2float(__ushort_as_half((unsigned short)(v & 0xffffu))); }
__device__ __forceinline__ float hi16(uint32_t v) { return __half2float(__ushort_as_half((unsigned short)(v >> 16))); }
__device__ __forceinline__ float sat16(float v) { return fminf(fmaxf(v, -65504.0f), 65504.0f); }   // finite saturation
__device__ __forceinline__ uint32_t pack16(float lo, float hi) {
  __half2 p = __floats2half2_rn(sat16(lo), sat16(hi));
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float act2f(act_t v) { return __half2float(v); }
__device__ __forceinline__ act_t f2act(float v) { return __float2half_rn(sat16(v)); }
#endif
// Packed fp32x2 FMA (sm_100 FFMA2): acc = a * b + acc on both halves with one instruction.
__device__ __forceinline__ void ffma2(float2& acc, const float2 a, const float2 b) {
  asm("{\n\t.reg .b64 ra, rb, rc;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%0, %1};\n\t"
      "fma.rn.f32x2 rc, ra, rb, rc;\n\t"
      "mov.b64 {%0, %1}, rc;\n\t}"
      : "+f"(acc.x), "+f"(acc.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
}
__device__ __forceinline__ float2 cvt16x2(uint32_t v) { return make_float2(lo16(v), hi16(v)); }

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// item of a global index in a ragged batch: the k with off[k] <= g < off[k+1] (off is a prefix array of B+1 entries, off[0] = 0)
__device__ __forceinline__ int find_item(const long long* __restrict__ off, int B, long long g) {
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(off + mid) <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Reduce (sum, sumsq) partials to (mean, rstd).  Called by a full warp; every lane returns the result.
// Deterministic (fixed order), accumulates in double.  (VQGAN GroupNorm(16) two-pass path.)
__device__ __forceinline__ float2 reduce_stats_warp(const float2* __restrict__ part, int slots, float inv_count,
                                                    float eps, int lane) {
  double s = 0.0, q = 0.0;
  for (int i = lane; i < slots; i += 32) {
    float2 v = __ldg(part + i);
    s += (double)v.x;
    q += (double)v.y;
  }
  s = warp_sum(s);
  q = warp_sum(q);
  double mean = s * (double)inv_count;
  double var = q * (double)inv_count - mean * mean;
  if (var < 0.0) var = 0.0;
  return make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
}

// ---- GroupNorm(1,C) statistics buffers ---------------------------------------------------------------------
// One buffer per normalised tensor: per sample `2 + slots` float2 entries
//   [0]            (mean, rstd)       -- final, written by the LAST producer tile of that sample
//   [1]            arrival counter (uint32 in .x; zero between launches: the last arriver resets it)
//   [2, 2+slots)   (sum, sumsq) partials, one per producer tile-warp
// The last arriver reduces the partials in slot order (double accumulation), so the result is deterministic
// whatever the arrival order.  Consumers read entry [0] only.
__device__ __forceinline__ const float2* stats_sample(const float2* base, int slots, int n) { return base + (size_t)n * (slots + 2); }
__device__ __forceinline__ float2* stats_sample(float2* base, int slots, int n) { return base + (size_t)n * (slots + 2); }

// Called by a full, converged warp; lane 0 carries this warp's (s, q).
__device__ __forceinline__ void stats_publish(float2* sb, int slots, int slot, float s, float q, float inv_count, float eps, int lane) {
  unsigned old = 0;
  if (lane == 0) {
    sb[2 + slot] = make_float2(s, q);
    __threadfence();
    old = atomicAdd(reinterpret_cast<unsigned*>(&sb[1]), 1u);
  }
  old = __shfl_sync(0xffffffffu, old, 0);
  if (old == (unsigned)(slots - 1)) {
    __threadfence();
    double ds = 0.0, dq = 0.0;
    for (int i = lane; i < slots; i += 32) {
      const float2 v = __ldcg(sb + 2 + i);
      ds += (double)v.x;
      dq += (double)v.y;
    }
    ds = warp_sum(ds);
    dq = warp_sum(dq);
    if (lane == 0) {
      const double mean = ds * (double)inv_count;
      double var = dq * (double)inv_count - mean * mean;
      if (var < 0.0) var = 0.0;
      sb[0] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
      *reinterpret_cast<unsigned*>(&sb[1]) = 0u;
    }
  }
}

// Run form: a block that produced `k` slots of one sample (each written with a plain store by lane 0 of the calling warp)
// announces them with ONE fence + atomic; the slots, and therefore the slot-ordered double-precision reduction of the last
// arriver, are exactly those of the per-tile protocol (results do not depend on how tiles are grouped into runs).  The fence +
// atomic round trip of a per-tile publish (2-3 us behind the block's own output stores) otherwise sits on the critical path
// of every tile.
__device__ __forceinline__ void stats_arrive_run(float2* sb, int slots, int k, float inv_count, float eps, int lane) {
  unsigned old = 0;
  if (lane == 0) {
    __threadfence();
    old = atomicAdd(reinterpret_cast<unsigned*>(&sb[1]), (unsigned)k);
  }
  old = __shfl_sync(0xffffffffu, old, 0);
  if (old + (unsigned)k == (unsigned)slots) {
    __threadfence();
    double ds = 0.0, dq = 0.0;
    for (int i = lane; i < slots; i += 32) {
      const float2 v = __ldcg(sb + 2 + i);
      ds += (double)v.x;
      dq += (double)v.y;
    }
    ds = warp_sum(ds);
    dq = warp_sum(dq);
    if (lane == 0) {
      const double mean = ds * (double)inv_count;
      double var = dq * (double)inv_count - mean * mean;
      if (var < 0.0) var = 0.0;
      sb[0] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
      *reinterpret_cast<unsigned*>(&sb[1]) = 0u;
    }
  }
}

// Branch-free GELU(erf): erf by Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7), straight-line code so the
// 16 independent elements of an epilogue chunk interleave.
__device__ __forceinline__ float gelu_erf_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = 1.0f - p * t * __expf(-z * z);      // erf(|x|/sqrt2)
  return 0.5f * x * (1.0f + copysignf(e, x));
}

// 256-bit global accesses (sm_100): one full 32-byte sector per lane instead of two 16-byte halves
__device__ __forceinline__ void stg_256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ void ldg_256(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}

}  // namespace ds
