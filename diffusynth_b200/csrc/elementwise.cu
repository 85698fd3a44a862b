// Bandwidth-bound elementwise kernels of the sampling path: the fused CFG + DDIM/DDPM update,
// q_sample, inpaint mask blend, layout/precision conversions, GroupNorm apply (+residual),
// GroupNorm(16) statistics + activation for the VQGAN, and the tiny time/condition linears.
#include "common.cuh"
#include "../../include/diffusynth_b200.h"

namespace ds {

// ---------------------------------------------------------------------------------------------
// K11: eps = eps_u + s (eps_c - eps_u);  x0 = (x - c0 eps) / c1;  x_prev = c2 x0 + c3 eps + c4 z
// model/DiffSynthSampler.py:320,327,337,343 -- same operation order, fp32.
// coef (device): {sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev-sigma^2), sigma, cfg_scale, -, -}
// ---------------------------------------------------------------------------------------------
__global__ void ddim_step_kernel(const float4* __restrict__ eps_u, const float4* __restrict__ eps_c,
                                 const float4* __restrict__ x, const float4* __restrict__ z,
                                 const float* __restrict__ coef, float4* __restrict__ out, long long n4) {
  pdl_enter();
  const float c0 = coef[0], c1 = coef[1], c2 = coef[2], c3 = coef[3], c4 = coef[4], s = coef[5];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 ec = __ldg(eps_c + i), xv = __ldg(x + i);
    float e[4] = {ec.x, ec.y, ec.z, ec.w};
    if (eps_u != nullptr) {
      float4 eu = __ldg(eps_u + i);
      const float u[4] = {eu.x, eu.y, eu.z, eu.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) e[j] = __fadd_rn(u[j], __fmul_rn(s, __fsub_rn(e[j], u[j])));
    }
    float zz[4] = {0.f, 0.f, 0.f, 0.f};
    if (z != nullptr) { float4 zv = __ldg(z + i); zz[0] = zv.x; zz[1] = zv.y; zz[2] = zv.z; zz[3] = zv.w; }
    const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float x0 = __fdiv_rn(__fsub_rn(xx[j], __fmul_rn(c0, e[j])), c1);
      o[j] = __fadd_rn(__fadd_rn(__fmul_rn(c2, x0), __fmul_rn(c3, e[j])), __fmul_rn(c4, zz[j]));
    }
    out[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// q_sample: a*x0 + b*noise (model/DiffSynthSampler.py:290-294); coef = {a, b}, or one {a, b} pair per sample when
// per_sample4 > 0 (= float4 vectors per sample: the reference gathers the coefficients per batch element, :17-22,290-293)
__global__ void q_sample_kernel(const float4* __restrict__ x0, const float4* __restrict__ noise, const float* __restrict__ coef,
                                float4* __restrict__ out, long long n4, long long per_sample4) {
  pdl_enter();
  float a = coef[0], b = coef[1];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    if (per_sample4 > 0) { const long long n = i / per_sample4; a = __ldg(coef + 2 * n); b = __ldg(coef + 2 * n + 1); }
    float4 p = __ldg(x0 + i), q = __ldg(noise + i);
    out[i] = make_float4(__fadd_rn(__fmul_rn(a, p.x), __fmul_rn(b, q.x)), __fadd_rn(__fmul_rn(a, p.y), __fmul_rn(b, q.y)),
                         __fadd_rn(__fmul_rn(a, p.z), __fmul_rn(b, q.z)), __fadd_rn(__fmul_rn(a, p.w), __fmul_rn(b, q.w)));
  }
}

// inpaint blend: img = m*(a*guide + b*noise) + (1-m)*img   (model/DiffSynthSampler.py:502-510);
// mask is [B,1,H,W] broadcast over the C channels (mask_c == 1) or [B,C,H,W] (mask_c == C: the reference's inpaint caller repeats
// its mask over the channels, inpaint_with_text.py:229-231); coef = {a, b} (a=1,b=0 reproduces the i==0 branch).
__global__ void mask_blend_kernel(const float* __restrict__ guide, const float* __restrict__ noise, const float* __restrict__ mask,
                                  const float* __restrict__ coef, float* __restrict__ img, int C, int mask_c, long long hw, long long total) {
  pdl_enter();
  const float a = coef[0], b = coef[1];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / (C * hw), p = i % hw;
    const float m = __ldg(mask_c == 1 ? mask + n * hw + p : mask + i);
    const float g = b == 0.f ? __fmul_rn(a, guide[i]) : __fadd_rn(__fmul_rn(a, guide[i]), __fmul_rn(b, noise[i]));
    img[i] = __fadd_rn(__fmul_rn(m, g), __fmul_rn(__fsub_rn(1.0f, m), img[i]));
  }
}

// fp32 NCHW -> bf16 NHWC with the channel count padded to Cp (zeros); and back.
__global__ void nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ in, act_t* __restrict__ out, int C, int Cp,
                                             long long hw, long long total_pix) {
  pdl_enter();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_pix * Cp; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % Cp);
    const long long pix = i / Cp, n = pix / hw, p = pix % hw;
    out[i] = f2act(c < C ? in[(n * C + c) * hw + p] : 0.f);
  }
}
// Fast form (Cp % 8 == 0): one thread per pixel; the C plane reads are coalesced across the warp (consecutive pixels of one
// plane) and each thread writes its pixel's Cp channels as 16-byte vectors, so a warp writes one contiguous 32*Cp*2-byte span.
__global__ void __launch_bounds__(256)
nchw_f32_to_nhwc_vec_kernel(const float* __restrict__ in, uint4* __restrict__ out, int C, int Cp8, long long hw, long long total_pix) {
  pdl_enter();
  for (long long pix = blockIdx.x * (long long)blockDim.x + threadIdx.x; pix < total_pix; pix += (long long)gridDim.x * blockDim.x) {
    const long long n = pix / hw, p = pix % hw;
    const float* src = in + n * C * hw + p;
    for (int v = 0; v < Cp8; ++v) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { const int c = 8 * v + j; f[j] = c < C ? __ldg(src + (long long)c * hw) : 0.f; }
      out[pix * Cp8 + v] = make_uint4(pack16(f[0], f[1]), pack16(f[2], f[3]), pack16(f[4], f[5]), pack16(f[6], f[7]));
    }
  }
}
__global__ void nhwc_bf16_to_nchw_f32_kernel(const act_t* __restrict__ in, float* __restrict__ out, int C, int Cp,
                                             long long hw, long long total) {
  pdl_enter();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i % hw, r = i / hw;
    const int c = (int)(r % C);
    const long long n = r / C;
    out[i] = act2f(in[(n * hw + p) * Cp + c]);
  }
}

// ---------------------------------------------------------------------------------------------
// GroupNorm(1,C) apply + residual:  out = (y - mean) * rstd * gamma[c] + beta[c] + x
// (the to_out[1] GroupNorm and the Residual of the attention block, diffusion_components.py:264,22-29)
// grid = (chunks, N); y/x/out bf16 NHWC with C % 8 == 0.
// ---------------------------------------------------------------------------------------------
// The host picks gridDim.x * blockDim.x as a multiple of C/8, so a thread always meets the same 8 channels: their folded
// scale (rstd*gamma) and shift (beta - mean*rstd*gamma) live in registers and the loop is two FMAs per value, four
// independent 16-byte vectors in flight per thread.
__global__ void __launch_bounds__(256)
gn_apply_residual_kernel(const uint4* __restrict__ y, const uint4* __restrict__ x, uint4* __restrict__ out,
                         const float2* __restrict__ stats, int slots,
                         const float* __restrict__ gamma, const float* __restrict__ beta, int C8,
                         long long vec_per_sample, int x_batch_mod) {
  pdl_enter();
  const int n = blockIdx.y;
  const float2 mr = __ldg(stats_sample(stats, slots, n));
  const float mean = mr.x, rstd = mr.y;
  const uint4* yb = y + (size_t)n * vec_per_sample;
  const uint4* xb = x ? x + (size_t)(x_batch_mod > 0 ? n % x_batch_mod : n) * vec_per_sample : nullptr;
  uint4* ob = out + (size_t)n * vec_per_sample;
  const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;          // a multiple of C8
  const int c0 = (int)(i0 % C8) * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = rstd * __ldg(gamma + c0 + j);
    sh[j] = fmaf(-mean, sc[j], __ldg(beta + c0 + j));
  }
  auto apply = [&](const uint4& yv, const uint4& xv) {
    const uint32_t yy[4] = {yv.x, yv.y, yv.z, yv.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w};
    uint32_t oo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      oo[j] = pack16(fmaf(lo16(yy[j]), sc[2 * j], sh[2 * j]) + lo16(xx[j]), fmaf(hi16(yy[j]), sc[2 * j + 1], sh[2 * j + 1]) + hi16(xx[j]));
    return make_uint4(oo[0], oo[1], oo[2], oo[3]);
  };
  long long i = i0;
  for (; i + 3 * stride < vec_per_sample; i += 4 * stride) {
    uint4 yv[4], xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      yv[u] = __ldg(yb + i + u * stride);
      xv[u] = xb ? __ldg(xb + i + u * stride) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) ob[i + u * stride] = apply(yv[u], xv[u]);
  }
  for (; i < vec_per_sample; i += stride) ob[i] = apply(__ldg(yb + i), xb ? __ldg(xb + i) : make_uint4(0, 0, 0, 0));
}

// ---------------------------------------------------------------------------------------------
// VQGAN GroupNorm(G groups, eps 1e-6) + activation as two passes (model/VQGAN.py:12-27,223-226):
//   group_stats: per (sample, chunk) partial (sum, sumsq) per group       grid = (chunks, N)
//   gn_act:      out = act((x - mean_g) * rstd_g * gamma + beta)          act: 0 none, 1 relu, 2 swish
// x bf16 NHWC with Cp channels stored (C real, Cp - C zero padding), C % G == 0.
// ---------------------------------------------------------------------------------------------
// 16-byte (8-channel) accesses: the host picks blockDim.x as a multiple of Cp/8, so a thread always meets the same 8 channels.
__global__ void group_stats_kernel(const act_t* __restrict__ x, float2* __restrict__ part, int C, int Cp, int G,
                                   long long hw, int chunks) {
  pdl_enter();
  extern __shared__ float s_acc[];   // [pixel lanes][Cp][2]: per-thread (sum, sumsq) of every channel, summed in fixed order (deterministic)
  const int n = blockIdx.y, chunk = blockIdx.x, cpg = C / G, C8 = Cp / 8;
  const long long per = (hw + chunks - 1) / chunks;
  const long long p0 = chunk * per, p1 = (p0 + per < hw) ? p0 + per : hw;
  const uint4* xb = reinterpret_cast<const uint4*>(x + (size_t)n * hw * Cp);
  const int tv = threadIdx.x % C8;                       // this thread's 8-channel vector inside a pixel
  const int tp = threadIdx.x / C8, pstride = blockDim.x / C8;
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s[j] = 0.f; q[j] = 0.f; }
  auto accumulate = [&](const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = lo16(w[j]), b = hi16(w[j]);
      s[2 * j] += a; q[2 * j] = fmaf(a, a, q[2 * j]);
      s[2 * j + 1] += b; q[2 * j + 1] = fmaf(b, b, q[2 * j + 1]);
    }
  };
  long long p = p0 + tp;
  for (; p + 3 * pstride < p1; p += 4 * pstride) {          // four independent loads in flight
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(xb + (p + u * pstride) * C8 + tv);
#pragma unroll
    for (int u = 0; u < 4; ++u) accumulate(v[u]);
  }
  for (; p < p1; p += pstride) accumulate(__ldg(xb + p * C8 + tv));
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = tv * 8 + j;
    s_acc[(tp * Cp + c) * 2] = s[j];
    s_acc[(tp * Cp + c) * 2 + 1] = q[j];
  }
  __syncthreads();
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    float gs = 0.f, gq = 0.f;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c)
      for (int t = 0; t < pstride; ++t) { gs += s_acc[(t * Cp + c) * 2]; gq += s_acc[(t * Cp + c) * 2 + 1]; }
    part[((size_t)n * G + g) * chunks + chunk] = make_float2(gs, gq);
  }
}

// grid = (gx, N) with gx * blockDim.x a multiple of Cp/8 (fixed 8 channels per thread: scale/shift in registers)
__global__ void gn_act_kernel(const act_t* __restrict__ x, act_t* __restrict__ out, const float2* __restrict__ part,
                              int chunks, const float* __restrict__ gamma, const float* __restrict__ beta, int C, int Cp, int G,
                              long long hw, float eps, int act) {
  pdl_enter();
  extern __shared__ float s_ab[];   // per channel scale, shift  [2*Cp]
  const int n = blockIdx.y, cpg = C / G, C8 = Cp / 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int g = warp; g < G; g += nwarps) {
    float2 mr = reduce_stats_warp(part + ((size_t)n * G + g) * chunks, chunks, 1.0f / (float)(cpg * hw), eps, lane);
    for (int c = g * cpg + lane; c < (g + 1) * cpg; c += 32) {
      const float a = mr.y * gamma[c];
      s_ab[2 * c] = a;
      s_ab[2 * c + 1] = beta[c] - mr.x * a;
    }
  }
  for (int c = C + threadIdx.x; c < Cp; c += blockDim.x) { s_ab[2 * c] = 0.f; s_ab[2 * c + 1] = 0.f; }
  __syncthreads();
  const long long total = hw * C8;                       // 16-byte vectors per sample
  const uint4* xb = reinterpret_cast<const uint4*>(x + (size_t)n * hw * Cp);
  uint4* ob = reinterpret_cast<uint4*>(out + (size_t)n * hw * Cp);
  const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int c0 = (int)(i0 % C8) * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = s_ab[2 * (c0 + j)]; sh[j] = s_ab[2 * (c0 + j) + 1]; }
  auto apply = [&](const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a = fmaf(lo16(w[j]), sc[2 * j], sh[2 * j]);
      float b = fmaf(hi16(w[j]), sc[2 * j + 1], sh[2 * j + 1]);
      if (act == 1) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
      else if (act == 2) { a = __fdividef(a, 1.f + __expf(-a)); b = __fdividef(b, 1.f + __expf(-b)); }
      o[j] = pack16(a, b);
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
  };
  long long i = i0;
  for (; i + 3 * stride < total; i += 4 * stride) {        // four independent vectors in flight
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(xb + i + u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) ob[i + u * stride] = apply(v[u]);
  }
  for (; i < total; i += stride) ob[i] = apply(__ldg(xb + i));
}

// x[n][p][c] += bias[n * bias_stride + c] in place (16-bit NHWC): the time embedding ResnetBlock adds between its two blocks
// (diffusion_components.py:97-100).  bias_stride 0 = one row for all samples.
__global__ void add_channel_bias_kernel(act_t* __restrict__ x, const float* __restrict__ bias, long long bias_stride, int C, long long per_sample /* hw*C/2 */,
                                        long long total) {
  pdl_enter();
  uint32_t* xv = reinterpret_cast<uint32_t*>(x);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / per_sample;
    const int c = (int)((i % (C / 2)) * 2);
    const float* b = bias + n * bias_stride + c;
    const uint32_t v = xv[i];
    xv[i] = pack16(lo16(v) + __ldg(b), hi16(v) + __ldg(b + 1));
  }
}

// out = a + b (bf16 NHWC), used for the VQGAN residual adds that are not fused into a conv epilogue
__global__ void add_bf16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out, long long n8) {
  pdl_enter();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 x = __ldg(a + i), y = __ldg(b + i);
    const uint32_t xx[4] = {x.x, x.y, x.z, x.w}, yy[4] = {y.x, y.y, y.z, y.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = pack16(lo16(xx[j]) + lo16(yy[j]), hi16(xx[j]) + hi16(yy[j]));
    out[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// VQGAN decoder head (model/VQGAN.py:394-398): ch0 softplus, ch1/ch2 tanh on (a + b); fp32 NCHW [N,3,H,W] in and out
// (a = final ResnetBlock conv, b = its nin_shortcut; both written as fp32 by the conv epilogue).
__global__ void decoder_head_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long hw, long long total) {
  pdl_enter();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / hw) % 3);
    const float v = a[i] + (b ? b[i] : 0.f);
    out[i] = c == 0 ? (v > 20.f ? v : log1pf(expf(v))) : tanhf(v);
  }
}

// ---------------------------------------------------------------------------------------------
// Tiny linears (time MLP, per-block time projections, condition projections):
//   out[n][o] = act_out(bias[o] + sum_k act_in(in[n][k]) * W[o][k])        act: 0 none, 1 GELU(erf), 2 SiLU (in), 3 tanh (out), 4 ReLU (out)
// One warp per output feature, looping over samples (the weight row stays in registers/L1).
// SinusoidalPositionEmbeddings (diffusion_components.py:42-56) is a separate small kernel.
// ---------------------------------------------------------------------------------------------
__global__ void linear_kernel(const float* __restrict__ in, long long in_stride, const float* __restrict__ W, const float* __restrict__ bias,
                              float* __restrict__ out, long long out_stride, int N, int K, int O, int act_in, int act_out) {
  pdl_enter();
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= O) return;
  const float* wr = W + (size_t)o * K;
  const float b = bias ? bias[o] : 0.f;
  for (int n = blockIdx.y; n < N; n += gridDim.y) {
    const float* xr = in + (size_t)n * in_stride;
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) {
      float v = xr[k];
      if (act_in == 1) v = gelu_erf(v);
      else if (act_in == 2) v = v / (1.0f + expf(-v));      // SiLU (ResnetBlock.mlp, diffusion_components.py:85-89)
      acc = fmaf(v, __ldg(wr + k), acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      float r = acc + b;
      if (act_out == 1) r = gelu_erf(r);
      else if (act_out == 3) r = tanhf(r);                 // ClapTextPooler
      else if (act_out == 4) r = fmaxf(r, 0.f);            // ClapProjectionLayer (projection_hidden_act = relu)
      out[(size_t)n * out_stride + o] = r;
    }
  }
}

// nn.Embedding lookup (ConditionalEmbedding with condition_type "instrument_family", diffusion_components.py:161,167)
__global__ void embedding_gather_kernel(const float* __restrict__ table, const long long* __restrict__ ids, float* __restrict__ out, int N, int D, int rows) {
  pdl_enter();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * D; i += gridDim.x * blockDim.x) {
    const int n = i / D, c = i - n * D;
    long long r = ids[n];
    r = r < 0 ? 0 : (r >= rows ? rows - 1 : r);
    out[i] = table[(size_t)r * D + c];
  }
}

__global__ void sinusoidal_kernel(const long long* __restrict__ t, float* __restrict__ out, int N, int dim) {
  pdl_enter();
  const int half = dim / 2;
  const float k = logf(10000.0f) / (float)(half - 1);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * half; i += gridDim.x * blockDim.x) {
    const int n = i / half, j = i % half;
    const float f = expf((float)j * -k);
    const float a = (float)t[n] * f;
    out[(size_t)n * dim + j] = sinf(a);
    out[(size_t)n * dim + half + j] = cosf(a);
  }
}

}  // namespace ds

using namespace ds;

extern "C" {

/* Fused CFG combine + DDIM/DDPM update (K11).  Replaces model/DiffSynthSampler.py:320-343.
   d_eps_u may be NULL (CFG == 1.0, :311-312); d_z may be NULL when sigma == 0.  n = elements. */
int ds_ddim_step(const float* d_eps_u, const float* d_eps_c, const float* d_x, const float* d_z, const float* d_coef,
                 float* d_out, long long n, void* stream) {
  DS_REQUIRE(d_eps_c && d_x && d_coef && d_out && n > 0 && n % 4 == 0, "ds_ddim_step: bad arguments (n=%lld must be a positive multiple of 4)", n);
  DS_CHECK_CUDA(launch_pdl(ddim_step_kernel, dim3(grid_for(n / 4, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, 
      (const float4*)d_eps_u, (const float4*)d_eps_c, (const float4*)d_x, (const float4*)d_z, d_coef, (float4*)d_out, n / 4));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_q_sample(const float* d_x0, const float* d_noise, const float* d_coef, float* d_out, long long n, long long per_sample,
                void* stream) {
  DS_REQUIRE(d_x0 && d_noise && d_coef && d_out && n > 0 && n % 4 == 0, "ds_q_sample: bad arguments");
  DS_REQUIRE(per_sample >= 0 && per_sample % 4 == 0 && (per_sample == 0 || n % per_sample == 0), "ds_q_sample: per_sample=%lld must divide n=%lld and be a multiple of 4", per_sample, n);
  DS_CHECK_CUDA(launch_pdl(q_sample_kernel, dim3(grid_for(n / 4, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const float4*)d_x0, (const float4*)d_noise, d_coef,
                                                                          (float4*)d_out, n / 4, per_sample / 4));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_mask_blend(const float* d_guide, const float* d_noise, const float* d_mask, int mask_channels, const float* d_coef, float* d_img,
                  int B, int C, long long hw, void* stream) {
  DS_REQUIRE(d_guide && d_noise && d_mask && d_coef && d_img && B > 0 && C > 0 && hw > 0, "ds_mask_blend: bad arguments");
  DS_REQUIRE(mask_channels == 1 || mask_channels == C, "ds_mask_blend: mask_channels=%d must be 1 or C=%d", mask_channels, C);
  const long long total = (long long)B * C * hw;
  DS_CHECK_CUDA(launch_pdl(mask_blend_kernel, dim3(grid_for(total, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, d_guide, d_noise, d_mask, d_coef, d_img, C, mask_channels, hw, total));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_add_channel_bias(void* d_x, const float* d_bias, long long bias_stride, int N, int C, long long hw, void* stream) {
  DS_REQUIRE(d_x && d_bias && N > 0 && C > 0 && C % 2 == 0 && hw > 0 && bias_stride >= 0, "ds_add_channel_bias: bad arguments");
  const long long per = hw * C / 2, total = per * N;
  DS_CHECK_CUDA(launch_pdl(add_channel_bias_kernel, dim3(grid_for(total, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, (act_t*)d_x, d_bias, bias_stride, C, per, total));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_nchw_f32_to_nhwc_bf16(const float* d_in, void* d_out, int N, int C, int Cp, long long hw, void* stream) {
  DS_REQUIRE(d_in && d_out && N > 0 && C > 0 && Cp >= C && hw > 0, "ds_nchw_f32_to_nhwc_bf16: bad arguments");
  if (Cp % 8 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0)
    DS_CHECK_CUDA(launch_pdl(nchw_f32_to_nhwc_vec_kernel, dim3(grid_for((long long)N * hw, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, d_in, (uint4*)d_out, C, Cp / 8, hw, (long long)N * hw));
  else
    DS_CHECK_CUDA(launch_pdl(nchw_f32_to_nhwc_bf16_kernel, dim3(grid_for((long long)N * hw * Cp, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, 
        d_in, (act_t*)d_out, C, Cp, hw, (long long)N * hw));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_nhwc_bf16_to_nchw_f32(const void* d_in, float* d_out, int N, int C, int Cp, long long hw, void* stream) {
  DS_REQUIRE(d_in && d_out && N > 0 && C > 0 && Cp >= C && hw > 0, "ds_nhwc_bf16_to_nchw_f32: bad arguments");
  const long long total = (long long)N * C * hw;
  DS_CHECK_CUDA(launch_pdl(nhwc_bf16_to_nchw_f32_kernel, dim3(grid_for(total, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const act_t*)d_in, d_out, C, Cp, hw, total));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_gn_apply_residual(const void* d_y, const void* d_x, void* d_out, const void* d_stats, int slots,
                         const float* d_gamma, const float* d_beta, int N, int C, long long hw, int x_batch_mod, void* stream) {
  DS_REQUIRE(d_y && d_out && d_stats && d_gamma && d_beta && N > 0 && C % 8 == 0 && hw > 0 && slots >= 0, "ds_gn_apply_residual: bad arguments");
  const long long vps = hw * C / 8;
  // threads per sample = gx * 256 must be a multiple of C/8 (see the kernel): gx is a multiple of m = C8 / gcd(C8, 256)
  const int C8 = C / 8;
  int g = C8, h256 = 256;
  while (h256) { const int t = g % h256; g = h256; h256 = t; }      // g = gcd(C8, 256)
  const int m = C8 / g;
  int gx = (int)((vps + 4 * 256 - 1) / (4 * 256));
  const int cap = (num_sms() * 8 + N - 1) / N;
  if (gx > cap) gx = cap;
  gx = (gx + m - 1) / m * m;
  if (gx < m) gx = m;
  DS_CHECK_CUDA(launch_pdl(gn_apply_residual_kernel, dim3(dim3(gx, N)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const uint4*)d_y, (const uint4*)d_x, (uint4*)d_out,
                                                                          (const float2*)d_stats, slots, d_gamma,
                                                                          d_beta, C / 8, vps, x_batch_mod));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_group_stats(const void* d_x, void* d_part, int N, int C, int Cp, int G, long long hw, int chunks, void* stream) {
  DS_REQUIRE(d_x && d_part && N > 0 && C > 0 && Cp >= C && Cp <= 1024 && G > 0 && C % G == 0 && chunks > 0, "ds_group_stats: bad arguments");
  DS_REQUIRE(Cp % 8 == 0, "ds_group_stats: Cp must be a multiple of 8");
  const int C8 = Cp / 8;
  const int block = C8 * 8;                    // 8 pixel lanes x Cp/8 channel vectors: few colliding shared atomics at the end
  DS_CHECK_CUDA(launch_pdl(group_stats_kernel, dim3(dim3(chunks, N)), dim3(block), (size_t)((size_t)8 * Cp * 2 * sizeof(float)), (cudaStream_t)stream, (const act_t*)d_x, (float2*)d_part,
                                                                                              C, Cp, G, hw, chunks));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_gn_act(const void* d_x, void* d_out, const void* d_part, int chunks, const float* d_gamma, const float* d_beta, int N, int C,
              int Cp, int G, long long hw, float eps, int act, void* stream) {
  DS_REQUIRE(d_x && d_out && d_part && d_gamma && d_beta && N > 0 && Cp % 2 == 0 && C % G == 0, "ds_gn_act: bad arguments");
  DS_REQUIRE(Cp % 8 == 0, "ds_gn_act: Cp must be a multiple of 8");
  const int C8 = Cp / 8;
  const long long total = hw * C8;
  int g = C8, h256 = 256;
  while (h256) { const int t = g % h256; g = h256; h256 = t; }      // gcd(C8, 256)
  const int m = C8 / g;                                             // gx must be a multiple of m
  int gx = (int)((total + 2 * 256 - 1) / (2 * 256));
  const int cap = (num_sms() * 8 + N - 1) / N;
  if (gx > cap) gx = cap;
  gx = (gx + m - 1) / m * m;
  if (gx < m) gx = m;
  DS_CHECK_CUDA(launch_pdl(gn_act_kernel, dim3(dim3(gx, N)), dim3(256), (size_t)((2 * Cp + 4) * sizeof(float)), (cudaStream_t)stream, 
      (const act_t*)d_x, (act_t*)d_out, (const float2*)d_part, chunks, d_gamma, d_beta, C, Cp, G, hw, eps, act));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_add_bf16(const void* d_a, const void* d_b, void* d_out, long long n, void* stream) {
  DS_REQUIRE(d_a && d_b && d_out && n > 0 && n % 8 == 0, "ds_add_bf16: bad arguments");
  DS_CHECK_CUDA(launch_pdl(add_bf16_kernel, dim3(grid_for(n / 8, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, (const uint4*)d_a, (const uint4*)d_b, (uint4*)d_out, n / 8));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_decoder_head(const float* d_a, const float* d_b, float* d_out, int N, long long hw, void* stream) {
  DS_REQUIRE(d_a && d_out && N > 0 && hw > 0, "ds_decoder_head: bad arguments");
  const long long total = (long long)N * 3 * hw;
  DS_CHECK_CUDA(launch_pdl(decoder_head_kernel, dim3(grid_for(total, 256, 8)), dim3(256), (size_t)(0), (cudaStream_t)stream, d_a, d_b, d_out, hw, total));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_linear(const float* d_in, long long in_stride, const float* d_w, const float* d_bias, float* d_out, long long out_stride, int N,
              int K, int O, int act_in, int act_out, void* stream) {
  DS_REQUIRE(d_in && d_w && d_out && N > 0 && K > 0 && O > 0, "ds_linear: bad arguments");
  const int wpb = 8;
  int gy = N < 16 ? N : 16;
  DS_CHECK_CUDA(launch_pdl(linear_kernel, dim3(dim3((O + wpb - 1) / wpb, gy)), dim3(wpb * 32), (size_t)(0), (cudaStream_t)stream, d_in, in_stride, d_w, d_bias, d_out, out_stride, N, K,
                                                                                      O, act_in, act_out));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

int ds_embedding_gather(const float* d_table, const long long* d_ids, float* d_out, int N, int D, int rows, void* stream) {
  DS_REQUIRE(d_table && d_ids && d_out && N > 0 && D > 0 && rows > 0, "ds_embedding_gather: bad arguments");
  DS_CHECK_CUDA(launch_pdl(embedding_gather_kernel, dim3(grid_for((long long)N * D, 256, 8)), dim3(256), (size_t)0, (cudaStream_t)stream, d_table, d_ids, d_out, N, D, rows));
  return DS_OK;
}

int ds_sinusoidal_embedding(const long long* d_t, float* d_out, int N, int dim, void* stream) {
  DS_REQUIRE(d_t && d_out && N > 0 && dim >= 4 && dim % 2 == 0, "ds_sinusoidal_embedding: bad arguments");
  DS_CHECK_CUDA(launch_pdl(sinusoidal_kernel, dim3(grid_for((long long)N * dim / 2, 128, 8)), dim3(128), (size_t)(0), (cudaStream_t)stream, d_t, d_out, N, dim));
  DS_CHECK_CUDA(cudaGetLastError());
  return DS_OK;
}

}  // extern "C"
