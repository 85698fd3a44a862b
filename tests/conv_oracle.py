"""Float64 restatement of the ds_conv_gemm and ds_dwconv7 contracts (include/diffusynth_b200.h), with per-element tolerances.

Both references take the operands exactly as the kernels read them -- 16-bit NHWC sources, the packed [Z, Cout_pad, K] weights,
the tap tables and views, the fp32 epilogue tables e1 / e2, entry 0 of the input statistics buffer -- and evaluate in float64
with torch on the operands' device (the GPU tests run it on the device, the CPU tests pin it to F.conv2d).

Tolerances.  A reference value v (before the 16-bit rounding of the output) comes with a gate g_v on |v_kernel - v| that sums
    accumulation   the kernel accumulates K = taps x Cin exact products (16-bit x 16-bit fits fp32) in fp32.  Each of the K
                   additions commits an error delta_j s_j with |delta_j| <= u32 = 2^-24 and |s_j| <= S = sum |x w|; modelled as
                   independent round-to-nearest noise (variance u32^2 / 3 s_j^2) this has sigma <= u32 sqrt(K / 3) S, and the gate
                   is 6 sigma: 6 u32 sqrt(K / 3) S, scaled by rstd where the GroupNorm fold multiplies it.
    fold           v = acc rstd + fma(-mean rstd, e1, e2) + sbias: four fp32 roundings, 4 u32 (|acc rstd| + |mean rstd e1| + |e2|
                   + |sbias|).
    GELU           the epilogue's erf is Abramowitz-Stegun 7.1.26 (|d erf| <= 1.5e-7, so |d GELU| <= 0.5 |x| 1.5e-7) evaluated
                   with approximate reciprocal / exp2 and an fp32 polynomial (16 u32 |x|); an error of the argument passes
                   through with the slope of GELU (<= 1.13).
    residual       one fp32 addition: u32 |v|.
The stored 16-bit output then adds one rounding: u16 |v| with u16 = 2^-11 (fp16) or 2^-8 (bf16), plus half the spacing of the
type's subnormals; fp16 outputs saturate at +-65504, and the reference saturates the same way.
Statistics (sum, sumsq per sample over the real channels and pixels, of the fp32 v): the element gates summed, plus fp32
summation (a thread's running sum over <= 128 columns, a 5-level warp tree, 8 warps: depth <= 150) 150 u32 sum |v|.  The
published (mean, rstd) follow by first-order propagation, plus their rounding to fp32.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
import torch.nn.functional as F

U32 = 2.0 ** -24
U_FP16, U_BF16 = 2.0 ** -11, 2.0 ** -8
FLOOR_FP16, FLOOR_BF16 = 2.0 ** -25, 2.0 ** -134        # half the subnormal spacing
FP16_MAX = 65504.0
SIGMAS = 6.0
STATS_DEPTH = 150
GELU_SLOPE = 1.13


def unit_roundoff(dtype) -> float:
    return U_FP16 if dtype == torch.float16 else U_BF16


def acc_gate(S: torch.Tensor, K: int) -> torch.Tensor:
    """6-sigma fp32 accumulation noise of K terms whose absolute sum is S."""
    return SIGMAS * U32 * math.sqrt(K / 3.0) * S


def gelu64(x: torch.Tensor) -> torch.Tensor:
    return 0.5 * x * (1.0 + torch.special.erf(x / math.sqrt(2.0)))


def _views(x: torch.Tensor, kind: str, Hin: int, Win: int):
    """The kernel's views of an NHWC source: the identity, or the four (row parity, column parity) views of a stride-2 conv."""
    if kind != "down":
        return [x]
    return [x[:, py::2, px::2] for py in range(2) for px in range(2)]


def _tap_sum(x, w, taps, kind, Hin, Win, Hg, Wg, per_sample):
    """acc[n, h, w, o] = sum over taps t and channels c of view_t(x)[n, h + dy, w + dx, c] * w[z, o, t*C + c] (out of the view: 0).
    x float64 NHWC [n, Hin, Win, C], w float64 [Z, Cout_pad, ntaps*C] (Z = n when per_sample); returns [n, G, Hg, Wg, Cout_pad]."""
    n, C = x.shape[0], x.shape[-1]
    G = len(taps)
    out = torch.zeros((n, G, Hg, Wg, w.shape[1]), dtype=torch.float64, device=x.device)
    views = [F.pad(v, (0, 0, 2, 2, 2, 2)) for v in _views(x, kind, Hin, Win)]
    for g in range(G):
        for t, (dy, dx, v) in enumerate(taps[g]):
            xs = views[v][:, 2 + dy:2 + dy + Hg, 2 + dx:2 + dx + Wg, :]
            wt = w[:, :, t * C:(t + 1) * C]                      # [Z, O, C]
            if per_sample:
                out[:, g] += torch.einsum("nhwc,noc->nhwo", xs, wt)
            else:
                out[:, g] += torch.einsum("nhwc,oc->nhwo", xs, wt[g])
    return out


def border_classes(Hg: int, Wg: int, ncls: int, device) -> torch.Tensor:
    """Border class of every GEMM-grid pixel: (top / middle / bottom) x 3 + (left / middle / right) for a 3x3, else 0."""
    if ncls != 9:
        return torch.zeros((Hg, Wg), dtype=torch.long, device=device)
    hh = torch.arange(Hg, device=device).view(-1, 1).expand(Hg, Wg)
    ww = torch.arange(Wg, device=device).view(1, -1).expand(Hg, Wg)
    rc = torch.where(hh == 0, 0, torch.where(hh == Hg - 1, 2, 1))
    cc = torch.where(ww == 0, 0, torch.where(ww == Wg - 1, 2, 1))
    return rc * 3 + cc


def conv_gemm_ref(src0, src1, weight, taps, kind, N, Hin, Win, e2, cout, e1=None, ncls=1, mean_rstd=None, sbias=None, act=0,
                  residual=None, src_batch_mod=0, per_sample_weights=False, samples: Optional[Sequence[int]] = None, chunk=None):
    """ds_conv_gemm in float64.  src0 16-bit NHWC [src_batch_mod or N, Hin, Win, C0]; src1 [N, Hin, Win, C1] or None; weight 16-bit
    [Z, Cout_pad, ntaps*(C0+C1)]; taps per group (dy, dx, view); kind 's1' / 'down' / 'up'; e1 / e2 fp32 [ncls, Cout_pad];
    mean_rstd fp32 [n_src, 2] = entry 0 of the statistics buffer of source 0 (indexed by n % src_batch_mod, like source 0);
    sbias [N, >= Cout]; residual 16-bit NHWC [N, Hg, Wg, Cout] (s1 / down).  samples: evaluate only these samples.
    Returns (v, gate) float64 [n, G, Hg, Wg, Cout]: the value before the output rounding and its gate (module docstring)."""
    dev = src0.device
    samples = list(range(N)) if samples is None else list(samples)
    Hg, Wg = (Hin // 2, Win // 2) if kind == "down" else (Hin, Win)
    C0 = src0.shape[-1]
    C1 = 0 if src1 is None else src1.shape[-1]
    K = len(taps[0]) * (C0 + C1)
    cls = border_classes(Hg, Wg, ncls, dev)
    e2c = e2.double()[cls][..., :cout]                                   # [Hg, Wg, Cout]
    e1c = e1.double()[cls][..., :cout] if e1 is not None else None
    vs, gs = [], []
    chunk = chunk or max(1, int(2e8 // (Hin * Win * max(C0 + C1, weight.shape[1]))))
    for i in range(0, len(samples), chunk):
        idx = torch.tensor(samples[i:i + chunk], device=dev)
        nsrc = idx % src_batch_mod if src_batch_mod > 0 else idx
        x = src0[nsrc].double()
        if src1 is not None:
            x = torch.cat([x, src1[idx].double()], dim=-1)
        w = weight[idx] if per_sample_weights else weight
        w = w.double()
        acc = _tap_sum(x, w, taps, kind, Hin, Win, Hg, Wg, per_sample_weights)[..., :cout]
        S = _tap_sum(x.abs(), w.abs(), taps, kind, Hin, Win, Hg, Wg, per_sample_weights)[..., :cout]
        if mean_rstd is not None:
            mr = mean_rstd[nsrc].double()
            mean, rstd = mr[:, 0].view(-1, 1, 1, 1, 1), mr[:, 1].view(-1, 1, 1, 1, 1)
        else:
            mean = torch.zeros((), dtype=torch.float64, device=dev)
            rstd = torch.ones((), dtype=torch.float64, device=dev)
        v = acc * rstd + e2c
        gate = acc_gate(S, K) * rstd
        mag = (acc * rstd).abs() + e2c.abs()
        if e1c is not None:
            v = v - mean * rstd * e1c
            mag = mag + (mean * rstd * e1c).abs()
        if sbias is not None:
            sb = sbias[idx, :cout].double().view(-1, 1, 1, 1, cout)
            v = v + sb
            mag = mag + sb.abs()
        gate = gate + 4 * U32 * mag
        if act == 1:
            gate = GELU_SLOPE * gate + (0.5 * 1.5e-7 + 16 * U32) * v.abs()
            v = gelu64(v)
        if residual is not None:
            assert kind != "up"
            v = v + residual[idx].double()[:, None, :, :, :cout]
            gate = gate + U32 * v.abs()
        vs.append(v)
        gs.append(gate)
    return torch.cat(vs), torch.cat(gs)


def interleave_up(t: torch.Tensor) -> torch.Tensor:
    """[n, 4, Hg, Wg, C] phases of the transposed conv -> [n, 2 Hg, 2 Wg, C] (phase g = (row parity, column parity))."""
    n, G, Hg, Wg, C = t.shape
    assert G == 4
    return t.view(n, 2, 2, Hg, Wg, C).permute(0, 3, 1, 4, 2, 5).reshape(n, 2 * Hg, 2 * Wg, C)


def out16_ref(v: torch.Tensor, gate: torch.Tensor, dtype):
    """Reference and gate of a value stored in the 16-bit type (fp16 saturates at +-65504)."""
    u = unit_roundoff(dtype)
    if dtype == torch.float16:
        v = v.clamp(-FP16_MAX, FP16_MAX)
    return v, (1 + u) * gate + u * v.abs() + (FLOOR_FP16 if dtype == torch.float16 else FLOOR_BF16)


def worst(got: torch.Tensor, ref: torch.Tensor, gate: torch.Tensor) -> float:
    """max over elements of |got - ref| / gate (<= 1 passes); NaN / inf in the output count as failures."""
    d = (got.double() - ref).abs() / gate
    d = torch.where(torch.isfinite(d), d, torch.full_like(d, float("inf")))
    return float(d.max()) if d.numel() else 0.0


def stats_ref(v: torch.Tensor, gate: torch.Tensor, count: int, eps: float):
    """Per-sample reference of the published statistics of v [n, ...] and their gates:
    (sum, sumsq, mean, rstd) each [n], and the gates in the same order."""
    n = v.shape[0]
    v, gate = v.reshape(n, -1), gate.reshape(n, -1)
    s, q = v.sum(1), (v * v).sum(1)
    a, a2 = v.abs().sum(1), (v * v).sum(1)
    gs = gate.sum(1) + STATS_DEPTH * U32 * a
    gq = (2 * v.abs() * gate + gate * gate).sum(1) + STATS_DEPTH * U32 * a2
    mean = s / count
    var = (q / count - mean * mean).clamp_min(0.0)
    rstd = 1.0 / torch.sqrt(var + eps)
    gm = gs / count + U32 * mean.abs() + 1e-30
    gvar = gq / count + 2 * mean.abs() * gm
    gr = 0.5 * rstd ** 3 * gvar + 2 * U32 * rstd
    return (s, q, mean, rstd), (gs, gq, gm, gr)


def check_stats(buf: torch.Tensor, samples, v, gate, count, eps) -> float:
    """Worst gate fraction of a statistics buffer float2 [N][2 + slots] against float64: the slot sums, the published (mean, rstd)
    of the given samples; the arrival counters must be back to zero (returns inf otherwise)."""
    b = buf[list(samples)].double()
    if float(buf[list(samples), 1].abs().max()) != 0.0:
        return float("inf")
    (s, q, m, r), (gs, gq, gm, gr) = stats_ref(v, gate, count, eps)
    got = [b[:, 2:, 0].sum(1), b[:, 2:, 1].sum(1), b[:, 0, 0], b[:, 0, 1]]
    return max(worst(x, y, g) for x, y, g in zip(got, (s, q, m, r), (gs, gq, gm, gr)))


# ------------------------------------------------------------------------------------------------------------------------------
# ds_dwconv7
# ------------------------------------------------------------------------------------------------------------------------------
def dwconv7_ref(src0, src1, weight, tbias, tbias_stride, N, H, W, src_batch_mod=0, samples: Optional[Sequence[int]] = None,
                chunk=None):
    """ds_dwconv7 in float64.  src0 16-bit NHWC [src_batch_mod or N, H, W, C0], src1 [N, H, W, C1] or None, weight fp32 [49, C]
    (tap-major), tbias fp32 rows of tbias_stride (one row read for every sample when tbias_stride = 0).
    The tensor-core kernel (H >= 16) multiplies by the weights rounded to the 16-bit operand type, the FFMA2 kernel (H < 16) by
    the fp32 weights.  Returns (v, gate) float64 NHWC [n, H, W, C] as conv_gemm_ref (50 accumulated terms: 49 taps + the bias)."""
    dev = src0.device
    samples = list(range(N)) if samples is None else list(samples)
    C = weight.shape[1]
    w = weight.to(src0.dtype) if H >= 16 else weight
    w = w.double().t().reshape(C, 1, 7, 7)
    tb = tbias.reshape(-1) if tbias_stride == 0 else tbias
    vs, gs = [], []
    chunk = chunk or max(1, int(1e8 // (H * W * C)))
    for i in range(0, len(samples), chunk):
        idx = torch.tensor(samples[i:i + chunk], device=dev)
        nsrc = idx % src_batch_mod if src_batch_mod > 0 else idx
        x = src0[nsrc].double()
        if src1 is not None:
            x = torch.cat([x, src1[idx].double()], dim=-1)
        x = x.permute(0, 3, 1, 2)
        b = (tb[:C].double().view(1, C).expand(len(idx), C) if tbias_stride == 0 else tb[idx, :C].double()).view(-1, C, 1, 1)
        v = F.conv2d(x, w, None, padding=3, groups=C) + b
        S = F.conv2d(x.abs(), w.abs(), None, padding=3, groups=C) + b.abs()
        gate = acc_gate(S, 50) + U32 * v.abs()
        vs.append(v.permute(0, 2, 3, 1))
        gs.append(gate.permute(0, 2, 3, 1))
    return torch.cat(vs), torch.cat(gs)


def dwconv7_grid(C: int, H: int, W: int, N: int, sms: int = 148) -> dict:
    """Work distribution of ds_dwconv7 (the grid rule of csrc/dwconv.cu, ds_dwconv7): the tensor-core kernel (H >= 16) runs gm x
    (C / 32) blocks, block b of a channel block walking items [b per_block, (b + 1) per_block) of the N x tiles (sample, tile)
    items; the FFMA2 kernel (H < 16) runs one block per (tile, channel block, sample)."""
    if H < 16:
        tiles = -(-W // 16) * -(-H // 8)
        return dict(kernel="ffma2", tiles=tiles, grid=tiles * (C // 32) * N, per_block=1, crosses_sample=False)
    tiles = -(-W // 16) * -(-H // 16)
    work = N * tiles
    gm = max(1, min(2 * sms // (C // 32), work))
    per = -(-work // gm)
    cross = any((b * per) // tiles != (min(b * per + per, work) - 1) // tiles for b in range(gm) if b * per < work)
    return dict(kernel="mma", tiles=tiles, grid=gm, per_block=per, crosses_sample=cross)
