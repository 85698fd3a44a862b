"""Host-side helpers over the C ABI: weight packing for the implicit-GEMM convolution
(ds_conv_gemm) and thin tensor-level wrappers of the other entry points.

Tensors are torch CUDA tensors used purely as device memory (PyTorch is plumbing here);
all arithmetic happens in the library's kernels.  Every call is enqueued on
``torch.cuda.current_stream()`` so it is captured by ``torch.cuda.graph``."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ConvGemmArgs, ConvGemmPlanInfo, check



def _act_dtype():
    return torch.float16 if _lib.load().ds_operand_dtype() == 1 else torch.bfloat16


ACT = _act_dtype()      # 16-bit storage / MMA operand dtype the library was built with (fp16 by default)
BF16 = ACT              # (historical alias)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------
# tile / blocking choices
# ------------------------------------------------------------------------------------------
def choose_tile(H: int, W: int) -> Tuple[int, int]:
    """(Hb, Wb) with Hb*Wb == 128 minimising padded area; ties -> wider tile (longer TMA rows)."""
    best = None
    for wb in (128, 64, 32, 16, 8, 4, 2, 1):
        hb = 128 // wb
        area = -(-W // wb) * wb * -(-H // hb) * hb
        if best is None or area < best[0]:
            best = (area, hb, wb)
    return best[1], best[2]


NARROW_BELOW = 74      # CTAs of the widest tiling at or below which choose_bn narrows the N tile (half of the 148 SMs)


def choose_bn(cout_pad: int, m_units: int = 1 << 30) -> int:
    """N-tile width (the rule of csrc/engine.cu choose_bn): the widest divisor of Cout_pad (<= 256), or -- when that tiling would leave
    more than half of the SMs idle (m_units = samples x groups x 128-pixel tiles) -- the widest divisor <= 64."""
    wide = next((bn for bn in range(256, 15, -16) if cout_pad % bn == 0), None)
    if wide is None:
        raise ValueError(cout_pad)
    if m_units * (cout_pad // wide) > NARROW_BELOW:
        return wide
    return next((bn for bn in (64, 32) if bn < wide and cout_pad % bn == 0), wide)


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


# ------------------------------------------------------------------------------------------
# conv weight packing  (all on the CPU, once per load_state_dict)
# ------------------------------------------------------------------------------------------
@dataclass
class PackedConv:
    """Device-side constant data of one ds_conv_gemm call site."""
    weight: torch.Tensor            # bf16 [groups, Cout_pad, K]
    e2: torch.Tensor                # f32 [ncls, Cout_pad]
    e1: Optional[torch.Tensor]      # f32 [ncls, Cout_pad] or None
    taps: List[List[Tuple[int, int, int]]]   # per group: (dy, dx, view)
    cin: int
    cout: int
    cout_pad: int
    ncls: int
    kind: str                       # "s1" (stride-1), "down" (4x4 s2), "up" (convT 4x4 s2)
    bn: int = 0

    def to(self, device):
        self.weight = self.weight.to(device)
        self.e2 = self.e2.to(device)
        if self.e1 is not None:
            self.e1 = self.e1.to(device)
        return self


def _border_tables(wk_fold_bf16: torch.Tensor, w_raw: torch.Tensor, beta: Optional[torch.Tensor],
                   bias: Optional[torch.Tensor], ksize: int, cout_pad: int):
    """e1[cls][o] = sum over taps valid in border class cls, and channels, of the (bf16-rounded, gamma-folded)
    weights; e2[cls][o] = bias[o] + sum_valid sum_c W[o,c,tap]*beta[c].  cls = rowclass*3 + colclass."""
    O = w_raw.shape[0]
    # sums in float64, rounded once (csrc/engine.cu packs the same tables the same way: the two paths agree bit for bit)
    wf = wk_fold_bf16.double()                      # [O, k, k, C]
    s1 = wf.sum(dim=3)                              # [O, k, k]
    s2 = (w_raw.permute(0, 2, 3, 1) * beta).double().sum(dim=3) if beta is not None else torch.zeros_like(s1)
    ncls = 9 if ksize == 3 else 1
    e1 = torch.zeros(ncls, cout_pad)
    e2 = torch.zeros(ncls, cout_pad)
    for cls in range(ncls):
        rc, cc = (cls // 3, cls % 3) if ksize == 3 else (1, 1)
        ky = [k for k in range(ksize) if not (ksize == 3 and ((rc == 0 and k == 0) or (rc == 2 and k == 2)))]
        kx = [k for k in range(ksize) if not (ksize == 3 and ((cc == 0 and k == 0) or (cc == 2 and k == 2)))]
        e1[cls, :O] = s1[:, ky][:, :, kx].sum(dim=(1, 2)).float()
        e2[cls, :O] = s2[:, ky][:, :, kx].sum(dim=(1, 2)).float()
        if bias is not None:
            e2[cls, :O] += bias
    return e1, e2, ncls


def pack_conv_s1(w: torch.Tensor, bias: Optional[torch.Tensor], gamma: Optional[torch.Tensor] = None,
                 beta: Optional[torch.Tensor] = None, cin_pad: Optional[int] = None) -> PackedConv:
    """Stride-1 'same' conv (1x1 or 3x3), optionally preceded by GroupNorm(1, Cin) whose affine
    (gamma, beta) is folded: gamma into the weights, beta into e2; the per-sample (mean, rstd) scalars are
    applied by the kernel epilogue through e1.  ``cin_pad``: stored channel count of the source (zero padded)."""
    O, Cin, k, _ = w.shape
    w = w.float()
    wk = w.permute(0, 2, 3, 1).contiguous()          # [O, ky, kx, C]
    wfold = (wk * gamma if gamma is not None else wk).to(BF16)
    cp = cin_pad or Cin
    cout_pad = pad16(O)
    e1, e2, ncls = _border_tables(wfold, w, beta, bias, k, cout_pad)
    wp = torch.zeros(cout_pad, k, k, cp, dtype=BF16)
    wp[:O, :, :, :Cin] = wfold
    taps = [[(ky - k // 2, kx - k // 2, 0) for ky in range(k) for kx in range(k)]]
    return PackedConv(weight=wp.reshape(1, cout_pad, k * k * cp).contiguous(), e2=e2,
                      e1=e1 if gamma is not None else None, taps=taps, cin=cp, cout=O, cout_pad=cout_pad,
                      ncls=ncls, kind="s1")


def pack_conv_down(w: torch.Tensor, bias: torch.Tensor, cin_pad: Optional[int] = None) -> PackedConv:
    """Conv2d(k=4, stride=2, padding=1): tap (ky,kx) reads input pixel (2h+ky-1, 2w+kx-1), i.e. parity view
    ((ky+1)%2, (kx+1)%2) at half-resolution offset floor((k-1)/2)."""
    O, Cin, k, _ = w.shape
    assert k == 4
    cp = cin_pad or Cin
    cout_pad = pad16(O)
    wp = torch.zeros(cout_pad, 4, 4, cp, dtype=BF16)
    wp[:O, :, :, :Cin] = w.float().permute(0, 2, 3, 1).to(BF16)
    taps = [[((ky - 1) // 2, (kx - 1) // 2, ((ky + 1) % 2) * 2 + (kx + 1) % 2) for ky in range(4) for kx in range(4)]]
    e2 = torch.zeros(1, cout_pad)
    e2[0, :O] = bias
    return PackedConv(weight=wp.reshape(1, cout_pad, 16 * cp).contiguous(), e2=e2, e1=None, taps=taps, cin=cp,
                      cout=O, cout_pad=cout_pad, ncls=1, kind="down")


def pack_conv_up(w: torch.Tensor, bias: torch.Tensor, cin_pad: Optional[int] = None) -> PackedConv:
    """ConvTranspose2d(k=4, stride=2, padding=1), weight [Cin, Cout, 4, 4]: output phase (py, px) is a 2x2
    conv of the input: py=0 uses ky=1 (dy=0), ky=3 (dy=-1); py=1 uses ky=0 (dy=+1), ky=2 (dy=0)."""
    Cin, O, k, _ = w.shape
    assert k == 4
    cp = cin_pad or Cin
    cout_pad = pad16(O)
    sel = {0: [(1, 0), (3, -1)], 1: [(0, 1), (2, 0)]}
    wp = torch.zeros(4, cout_pad, 4, cp, dtype=BF16)
    taps = []
    wf = w.float()
    for py in range(2):
        for px in range(2):
            g, tl, t = py * 2 + px, [], 0
            for ky, dy in sel[py]:
                for kx, dx in sel[px]:
                    wp[g, :O, t, :Cin] = wf[:, :, ky, kx].t().to(BF16)
                    tl.append((dy, dx, 0))
                    t += 1
            taps.append(tl)
    e2 = torch.zeros(1, cout_pad)
    e2[0, :O] = bias
    return PackedConv(weight=wp.reshape(4, cout_pad, 4 * cp).contiguous(), e2=e2, e1=None, taps=taps, cin=cp,
                      cout=O, cout_pad=cout_pad, ncls=1, kind="up")


# ------------------------------------------------------------------------------------------
# conv call construction
# ------------------------------------------------------------------------------------------
@dataclass
class Stats:
    """GroupNorm(1,C) statistics buffer of one tensor: float2 [N][2 + slots] (see csrc/common.cuh):
    [n][0] = (mean, rstd) published by the producer's last tile, [n][1] = arrival counter, then the partials.
    count = elements per sample."""
    buf: torch.Tensor
    slots: int
    count: int


def new_stats(N: int, slots: int, count: int, device) -> Stats:
    return Stats(torch.zeros((N, slots + 2, 2), dtype=torch.float32, device=device), slots, count)


def given_stats(mean: torch.Tensor, rstd: torch.Tensor, count: int, device="cuda") -> Stats:
    """A statistics buffer carrying externally computed (mean, rstd) per sample (tests)."""
    buf = torch.zeros((mean.shape[0], 2, 2), dtype=torch.float32)
    buf[:, 0, 0], buf[:, 0, 1] = mean, rstd
    return Stats(buf.to(device), 0, count)


def conv_args(pc: PackedConv, src0: torch.Tensor, src1: Optional[torch.Tensor], N: int, Hin: int, Win: int,
              out: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None,
              stats_in: Optional[Stats] = None, eps: float = 1e-5, sbias: Optional[torch.Tensor] = None,
              act: int = 0, residual: Optional[torch.Tensor] = None, want_stats: bool = False,
              src_batch_mod: int = 0, weight_override: Optional[torch.Tensor] = None,
              per_sample_weights: bool = False, device=None, wide_tiles: bool = False) -> Tuple[ConvGemmArgs, Optional[Stats], list]:
    """Build the argument block of one ds_conv_gemm call.  ``src*`` bf16 NHWC [N, Hin, Win, C].
    Returns (args, stats_out, keepalive)."""
    a = ConvGemmArgs()
    C0 = src0.shape[-1]
    C1 = 0 if src1 is None else src1.shape[-1]
    assert C0 + C1 == pc.cin, (C0, C1, pc.cin)
    a.d_src0, a.d_src1 = _ptr(src0), _ptr(src1)
    a.C0, a.C1, a.N, a.src_batch_mod = C0, C1, N, src_batch_mod
    if pc.kind == "down":
        Hg, Wg = Hin // 2, Win // 2
        a.Hv, a.Wv = Hg, Wg
        a.view_sn, a.view_sh, a.view_sw = Hin * Win, 2 * Win, 2
        for v in range(4):
            a.view_off[v] = (v // 2) * Win + (v % 2)
            # odd input sizes: the even-parity view holds one more column / row than the odd one (the conv's last tap
            # still reads input column 2*Wg = Win-1)
            a.view_hv[v], a.view_wv[v] = (Hin - v // 2 + 1) // 2, (Win - v % 2 + 1) // 2
        a.num_views = 4
        Ho, Wo = Hg, Wg
    else:
        Hg, Wg = Hin, Win
        a.Hv, a.Wv = Hin, Win
        a.view_sn, a.view_sh, a.view_sw = Hin * Win, Win, 1
        a.num_views = 1
        Ho, Wo = (2 * Hin, 2 * Win) if pc.kind == "up" else (Hin, Win)
    a.H, a.W = Hg, Wg
    a.Hb, a.Wb = choose_tile(Hg, Wg)
    w = weight_override if weight_override is not None else pc.weight
    a.d_weight = _ptr(w)
    a.Cout_pad, a.Cout = pc.cout_pad, pc.cout
    a.BN = pc.bn or (choose_bn(pc.cout_pad) if wide_tiles else choose_bn(pc.cout_pad, N * len(pc.taps) * (-(-Hg // a.Hb)) * (-(-Wg // a.Wb))))
    a.BK = 64 if (C0 % 64 == 0 and C1 % 64 == 0) else 32
    a.ntaps, a.groups = len(pc.taps[0]), len(pc.taps)
    a.per_sample_weights = 1 if per_sample_weights else 0
    for g, tl in enumerate(pc.taps):
        for t, (dy, dx, v) in enumerate(tl):
            a.taps[g][t].dy, a.taps[g][t].dx, a.taps[g][t].view = dy, dx, v
    if stats_in is not None:
        assert pc.e1 is not None
        a.d_stats_in, a.stats_in_slots = _ptr(stats_in.buf), stats_in.slots
        a.d_e1 = _ptr(pc.e1)
    a.eps = eps
    a.d_e2, a.ncls = _ptr(pc.e2), pc.ncls
    if sbias is not None:
        a.d_sbias, a.sbias_stride = _ptr(sbias), sbias.stride(0)
    a.act = act
    if residual is not None:
        Cr = residual.shape[-1]
        a.d_residual, a.res_sn, a.res_sh, a.res_sw = _ptr(residual), Ho * Wo * Cr, Wo * Cr, Cr
    if out is not None:
        Co = out.shape[-1]
        a.d_out = _ptr(out)
        if pc.kind == "up":
            # the output may be a larger zero-initialised map [N, Hp, Wp, Co] (pad_to_match, diffusion_components.py:210-232:
            # the upsampled map sits at (delta // 2) from the top/left, the remainder stays zero)
            Hp, Wp = out.shape[1], out.shape[2]
            assert Hp >= Ho and Wp >= Wo, (Hp, Wp, Ho, Wo)
            org = ((Hp - Ho) // 2) * Wp + (Wp - Wo) // 2
            a.out_sn, a.out_sh, a.out_sw = Hp * Wp * Co, 2 * Wp * Co, 2 * Co
            for g in range(4):
                a.out_goff[g] = (org + (g // 2) * Wp + (g % 2)) * Co
        else:
            a.out_sn, a.out_sh, a.out_sw = Ho * Wo * Co, Wo * Co, Co
    a.d_out_f32_nchw = _ptr(out_f32)
    keep = [src0, src1, w, pc, stats_in, sbias, residual, out, out_f32]
    st = None
    if want_stats:
        slots = _lib.load().ds_conv_gemm_stats_slots(C.byref(a))
        st = new_stats(N, slots, Ho * Wo * pc.cout, src0.device)
        a.d_stats_out = _ptr(st.buf)
        a.stats_out_inv_count = 1.0 / st.count
        keep.append(st)
    return a, st, keep


def conv_cost(a: ConvGemmArgs, pc: PackedConv) -> Tuple[str, float, float]:
    """(kernel family, algorithmic FLOPs, algorithmic HBM bytes) of one ds_conv_gemm call: 2 FLOP per MAC over the real channels,
    every operand moved once (activations in, weights, residual, output)."""
    cin = a.C0 + a.C1
    flops = 2.0 * a.N * a.groups * a.H * a.W * a.Cout * a.ntaps * cin
    n_in = a.src_batch_mod if a.src_batch_mod > 0 else a.N
    hin, win = (2 * a.H, 2 * a.W) if pc.kind == "down" else (a.H, a.W)
    by = n_in * hin * win * a.C0 * 2.0 + a.N * hin * win * a.C1 * 2.0
    by += (a.N if a.per_sample_weights else a.groups) * a.Cout_pad * a.ntaps * cin * 2.0
    out_px = a.N * a.groups * a.H * a.W
    if a.d_out:
        by += out_px * a.Cout * 2.0
    if a.d_out_f32_nchw:
        by += out_px * a.Cout * 4.0
    if a.d_residual:
        by += out_px * a.Cout * 2.0
    fam = "conv3x3" if (pc.kind == "s1" and a.ntaps == 9) else "conv1x1" if pc.kind == "s1" else "conv4x4s2" if pc.kind == "down" else "convT4x4s2"
    return fam, flops, by


def conv_plan(a: ConvGemmArgs) -> dict:
    """The launch ds_conv_gemm makes for this argument block (ds_conv_gemm_plan; host only), plus the mean number of work items
    per CTA (per CTA pair when cg = 2)."""
    info = ConvGemmPlanInfo()
    check(_lib.load().ds_conv_gemm_plan(C.byref(a), C.byref(info)), "ds_conv_gemm_plan")
    plan = {name: getattr(info, name) for name, _ in ConvGemmPlanInfo._fields_}
    plan["items_per_cta"] = plan["num_tiles"] / (plan["grid"] // plan["cg"])
    return plan


def run_conv(a: ConvGemmArgs, reference: bool = False) -> None:
    lib = _lib.load()
    fn = lib.ds_conv_gemm_reference if reference else lib.ds_conv_gemm
    check(fn(C.byref(a), _stream()), "ds_conv_gemm")


# ------------------------------------------------------------------------------------------
# thin wrappers
# ------------------------------------------------------------------------------------------
def ddim_step(eps_u, eps_c, x, z, coef, out):
    check(_lib.load().ds_ddim_step(_ptr(eps_u), _ptr(eps_c), _ptr(x), _ptr(z), _ptr(coef), _ptr(out), x.numel(), _stream()),
          "ds_ddim_step")


def q_sample(x0, noise, coef, out, per_sample: int = 0):
    """coef [2] (one (a, b) pair) or [B, 2] with per_sample = elements per sample."""
    check(_lib.load().ds_q_sample(_ptr(x0), _ptr(noise), _ptr(coef), _ptr(out), x0.numel(), per_sample, _stream()), "ds_q_sample")


def normalize_mask(mask: torch.Tensor, shape, device) -> torch.Tensor:
    """The reference multiplies ``mask * img`` (DiffSynthSampler.py:506,510), i.e. any mask broadcastable to [B,C,H,W]
    works there; its callers pass [B,1,H,W] (track_maker.py:252) and [B,C,H,W] (inpaint_with_text.py:229-231).
    Returns a contiguous fp32 [B,1,H,W] or [B,C,H,W] tensor."""
    B, Cc, H, W = shape
    m = mask.to(device, torch.float32)
    while m.dim() < 4:
        m = m.unsqueeze(0)
    mc = 1 if m.shape[1] == 1 else Cc
    return m.expand(B, mc, H, W).contiguous()


def mask_blend(guide, noise, mask, coef, img):
    B, Cc, H, W = img.shape
    assert mask.shape[0] == B and mask.shape[1] in (1, Cc) and tuple(mask.shape[2:]) == (H, W) and mask.is_contiguous(), tuple(mask.shape)
    check(_lib.load().ds_mask_blend(_ptr(guide), _ptr(noise), _ptr(mask), mask.shape[1], _ptr(coef), _ptr(img), B, Cc, H * W, _stream()),
          "ds_mask_blend")


def dwconv7_stats(N, C, H, W, device) -> Stats:
    return new_stats(N, _lib.load().ds_dwconv7_stats_slots(C, H, W), H * W * C, device)


def dwconv7(src0, src1, weight, tbias, tbias_stride, out, N, H, W, stats: Optional[Stats] = None, src_batch_mod=0, eps=1e-5) -> None:
    C0 = src0.shape[-1]
    C1 = 0 if src1 is None else src1.shape[-1]
    check(_lib.load().ds_dwconv7(_ptr(src0), _ptr(src1), C0, C1, src_batch_mod, _ptr(weight), _ptr(tbias), tbias_stride, _ptr(out),
                                 _ptr(stats.buf) if stats else None, eps, N, H, W, _stream()), "ds_dwconv7")


def linear(inp, w, bias, out, act_in=0, act_out=0):
    N, K = inp.shape
    O = w.shape[0]
    check(_lib.load().ds_linear(_ptr(inp), inp.stride(0), _ptr(w), _ptr(bias), _ptr(out), out.stride(0), N, K, O, act_in,
                                act_out, _stream()), "ds_linear")
