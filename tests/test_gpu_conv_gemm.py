"""tcgen05 implicit-GEMM convolution (ds_conv_gemm) against (a) the kernel contract evaluated by torch on the
CPU (the oracle for this op: fp32 conv of the bf16-rounded operands) and (b) the CUDA-core cross-check kernel."""
import pytest
import torch
import torch.nn.functional as F

from oracle import cases
from tests.gpu_util import EPS16, bf, nchw, nhwc, rel
from tests.test_host_packing import contract

pytestmark = pytest.mark.gpu

# output rounding of the 16-bit storage type: EPS16/2 relative per element (fp16: 2^-12, bf16: 2^-9)
TOL = EPS16


def _run(pc, srcs, N, H, W, reference=False, **kw):
    from diffusynth_b200 import ops
    pc.to("cuda")
    a, st, keep = ops.conv_args(pc, srcs[0], srcs[1] if len(srcs) > 1 else None, N, H, W, **kw)
    ops.run_conv(a, reference=reference)
    torch.cuda.synchronize()
    return st


# Small jobs (these are all far below the 148 SMs) run narrow N tiles and one work item per CTA: (BN, cg, pair_flat) each case
# runs, from the planner query.  Wide N tiles and persistent runs of many items per CTA: tests/test_gpu_conv_scale.py.
PLAIN_PLANS = {
    (64, 64, 3, 16, 8, 2): (32, 2, 1),
    (96, 192, 3, 32, 16, 2): (64, 2, 0),
    (128, 96, 1, 16, 16, 3): (32, 1, 0),
    (192, 384, 3, 16, 8, 1): (64, 1, 0),
    (192, 384, 3, 16, 8, 4): (64, 2, 1),
    (128, 96, 3, 16, 24, 3): (32, 1, 0),
    (64, 768, 1, 16, 8, 2): (64, 1, 0),
    (96, 96, 3, 128, 64, 2): (96, 2, 0),
    (32, 32, 3, 128, 24, 1): (32, 2, 0),
    (64, 48, 3, 20, 12, 2): (48, 1, 0),
    (96, 192, 3, 64, 32, 2): (64, 2, 0),
    (64, 64, 3, 20, 40, 3): (32, 1, 0),
    (128, 256, 3, 128, 64, 1): (64, 2, 0),
}


@pytest.mark.parametrize("cin,cout,k,H,W,N", [
    (64, 64, 3, 16, 8, 2),        # BK=64 (SWIZZLE_128B), one tile per sample: the two-CTA pair spans both samples
    (96, 192, 3, 32, 16, 2),      # BK=32 (SWIZZLE_64B), 4 m-tiles
    (128, 96, 1, 16, 16, 3),      # 1x1
    (192, 384, 3, 16, 8, 1),      # six narrow n-tiles (BN=64), one CTA per tile
    (192, 384, 3, 16, 8, 4),      # one M-tile per sample: the two-CTA pairs span consecutive samples
    (128, 96, 3, 16, 24, 3),      # three M-tiles per sample, odd sample count: falls back to one CTA per tile
    (64, 768, 1, 16, 8, 2),       # 1x1 with twelve narrow n-tiles (BN=64), two CTAs per SM
    (96, 96, 3, 128, 64, 2),      # full-resolution level-0 shape, 64 m-tiles per sample
    (32, 32, 3, 128, 24, 1),      # width not a multiple of the preferred tile
    (64, 48, 3, 20, 12, 2),       # ragged: partial tiles in both directions
    (96, 192, 3, 64, 32, 2),      # BK=32 with several K-blocks per stage
    (64, 64, 3, 20, 40, 3),       # ragged, W > 32
    (128, 256, 3, 128, 64, 1),    # BK=64, 64 tiles per sample, four n-tiles: up to two items per CTA pair
])
def test_plain_conv(cin, cout, k, H, W, N):
    from diffusynth_b200 import ops
    x = cases.randn((N, cin, H, W), 1)
    w, b = cases.randn((cout, cin, k, k), 2) * (1.0 / (cin * k * k) ** 0.5), cases.randn((cout,), 3)
    pc = ops.pack_conv_s1(w, b)
    out = torch.zeros((N, H, W, cout), dtype=ops.ACT, device="cuda")
    a, _, _ = ops.conv_args(pc.to("cuda"), nhwc(x), None, N, H, W, out=out)
    plan = ops.conv_plan(a)
    assert (plan["BN"], plan["cg"], plan["pair_flat"]) == PLAIN_PLANS[(cin, cout, k, H, W, N)]
    _run(pc, [nhwc(x)], N, H, W, out=out)
    ref = F.conv2d(bf(x), bf(w), b, padding=k // 2)
    assert rel(nchw(out), ref) < TOL
    out2 = torch.zeros_like(out)
    _run(pc, [nhwc(x)], N, H, W, reference=True, out=out2)
    assert rel(nchw(out2), ref) < TOL
    assert rel(nchw(out), nchw(out2)) < TOL


def test_convnext_conv1_fold_gelu_stats_concat():
    """Two concatenated sources, GroupNorm(1,C) folded, GELU, and the (sum, sumsq) partials for the next norm."""
    from diffusynth_b200 import ops
    N, H, W = 2, 16, 32
    x0, x1 = cases.randn((N, 96, H, W), 4) + 0.5, cases.randn((N, 192, H, W), 5) * 1.7
    w, b = cases.randn((192, 288, 3, 3), 6) * 0.02, cases.randn((192,), 7) * 0.1
    gamma, beta = 1 + 0.2 * cases.randn((288,), 8), 0.2 * cases.randn((288,), 9)
    pc = ops.pack_conv_s1(w, b, gamma, beta)
    xb = torch.cat([bf(x0), bf(x1)], 1)
    # statistics of the (bf16-stored) source as one partial slot per sample
    st = ops.given_stats(xb.mean(dim=(1, 2, 3)), (xb.var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt(), 288 * H * W)
    out = torch.zeros((N, H, W, 192), dtype=ops.ACT, device="cuda")
    so = _run(pc, [nhwc(x0), nhwc(x1)], N, H, W, out=out, stats_in=st, act=1, want_stats=True)
    ref = F.gelu(F.conv2d(F.group_norm(xb, 1, gamma, beta, 1e-5), w, b, padding=1))
    got = nchw(out)
    assert rel(got, ref) < 1.5 * TOL
    # published statistics of the output: partial slots sum to the fp32 totals; entry 0 = (mean, rstd); counter reset
    buf = so.buf.double().cpu()
    s = buf[:, 2:].sum(dim=1)
    assert torch.allclose(s[:, 0], ref.double().sum(dim=(1, 2, 3)), rtol=2e-3, atol=4.0)
    assert torch.allclose(s[:, 1], (ref.double() ** 2).sum(dim=(1, 2, 3)), rtol=4e-3)
    assert so.count == 192 * H * W
    assert torch.allclose(buf[:, 0, 0], ref.double().mean(dim=(1, 2, 3)), rtol=2e-3, atol=1e-4)
    assert torch.allclose(buf[:, 0, 1], (ref.double().var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt(), rtol=2e-3)
    assert float(so.buf[:, 1].abs().max()) == 0.0
    # second launch into the same buffer (counter must have reset itself): identical statistics
    first = so.buf.clone()
    a2, so2, _ = ops.conv_args(pc, nhwc(x0), nhwc(x1), N, H, W, out=out, stats_in=st, act=1, want_stats=True)
    a2.d_stats_out = so.buf.data_ptr()
    ops.run_conv(a2)
    torch.cuda.synchronize()
    assert torch.equal(first, so.buf)


@pytest.mark.parametrize("H,W", [(16, 8), (8, 64)])
def test_conv2_residual_and_contract_cross_check(H, W):
    from diffusynth_b200 import ops
    N = 2
    x, r = cases.randn((N, 128, H, W), 10) * 2 + 1, cases.randn((N, 64, H, W), 11)
    w, b = cases.randn((64, 128, 3, 3), 12) * 0.03, cases.randn((64,), 13) * 0.1
    gamma, beta = 1 + 0.2 * cases.randn((128,), 14), 0.2 * cases.randn((128,), 15)
    pc = ops.pack_conv_s1(w, b, gamma, beta)
    xb = bf(x)
    st = ops.given_stats(xb.mean(dim=(1, 2, 3)), (xb.var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt(), 128 * H * W)
    out = torch.zeros((N, H, W, 64), dtype=ops.ACT, device="cuda")
    _run(pc, [nhwc(x)], N, H, W, out=out, stats_in=st, residual=nhwc(r))
    ref = F.conv2d(F.group_norm(xb, 1, gamma, beta, 1e-5), w, b, padding=1) + bf(r)
    assert rel(nchw(out), ref) < 1.5 * TOL
    pc_cpu = ops.pack_conv_s1(w, b, gamma, beta)
    for n in range(N):
        mean, var = xb[n].mean(), xb[n].var(unbiased=False)
        c = contract(pc_cpu, [x[n:n + 1]], "s1", (mean, (var + 1e-5).rsqrt()), residual=bf(r[n:n + 1]))
        assert rel(nchw(out)[n:n + 1], c) < TOL


def test_downsample_and_upsample():
    from diffusynth_b200 import ops
    N, H, W = 2, 32, 16
    x = cases.randn((N, 96, H, W), 16)
    w, b = cases.randn((96, 96, 4, 4), 17) * 0.03, cases.randn((96,), 18)
    pc = ops.pack_conv_down(w, b)
    out = torch.zeros((N, H // 2, W // 2, 96), dtype=ops.ACT, device="cuda")
    _run(pc, [nhwc(x)], N, H, W, out=out)
    assert rel(nchw(out), F.conv2d(bf(x), bf(w), b, stride=2, padding=1)) < TOL
    wt = cases.randn((96, 64, 4, 4), 19) * 0.05
    bt = cases.randn((64,), 20)
    pcu = ops.pack_conv_up(wt, bt)
    outu = torch.zeros((N, 2 * H, 2 * W, 64), dtype=ops.ACT, device="cuda")
    _run(pcu, [nhwc(x)], N, H, W, out=outu)
    assert rel(nchw(outu), F.conv_transpose2d(bf(x), bf(wt), bt, stride=2, padding=1)) < TOL


@pytest.mark.parametrize("H,W", [(16, 7), (9, 5), (32, 13)])
def test_downsample_odd_sizes_and_padded_upsample(H, W):
    """Odd input sizes of the 4x4 stride-2 conv (per-view extents), and the ConvTranspose written into a larger
    zero map at pad_to_match's offset (diffusion_components.py:210-232)."""
    from diffusynth_b200 import ops
    N = 2
    x = cases.randn((N, 96, H, W), 26)
    w, b = cases.randn((96, 96, 4, 4), 17) * 0.03, cases.randn((96,), 18)
    pc = ops.pack_conv_down(w, b)
    ref = F.conv2d(bf(x), bf(w), b, stride=2, padding=1)
    out = torch.zeros((N, H // 2, W // 2, 96), dtype=ops.ACT, device="cuda")
    _run(pc, [nhwc(x)], N, H, W, out=out)
    assert tuple(ref.shape[2:]) == (H // 2, W // 2) and rel(nchw(out), ref) < TOL
    out2 = torch.zeros_like(out)
    _run(pc, [nhwc(x)], N, H, W, reference=True, out=out2)
    assert rel(nchw(out2), ref) < TOL
    # up: the half-size map back to (2*(H//2), 2*(W//2)), placed in an H x W map
    y = cases.randn((N, 96, H // 2, W // 2), 27)
    wt, bt = cases.randn((96, 64, 4, 4), 19) * 0.05, cases.randn((64,), 20)
    pcu = ops.pack_conv_up(wt, bt)
    outu = torch.zeros((N, H, W, 64), dtype=ops.ACT, device="cuda")
    _run(pcu, [nhwc(y)], N, H // 2, W // 2, out=outu)
    up = F.conv_transpose2d(bf(y), bf(wt), bt, stride=2, padding=1)
    dh, dw = H - up.shape[2], W - up.shape[3]
    refu = F.pad(up, (dw // 2, dw - dw // 2, dh // 2, dh - dh // 2))
    assert rel(nchw(outu), refu) < TOL
    assert float(nchw(outu)[:, :, :, W - (dw - dw // 2):].abs().max() if dw else 0.0) == 0.0


def test_final_conv_fp32_nchw_and_batch_mod():
    from diffusynth_b200 import ops
    N, H, W = 4, 16, 8
    x = cases.randn((2, 96, H, W), 21)          # 2 stored samples serve 4 logical ones (CFG doubling)
    w, b = cases.randn((4, 96, 3, 3), 22) * 0.05, cases.randn((4,), 23)
    pc = ops.pack_conv_s1(w, b)
    out = torch.zeros((N, 4, H, W), dtype=torch.float32, device="cuda")
    _run(pc, [nhwc(x)], N, H, W, out_f32=out, src_batch_mod=2)
    ref = F.conv2d(bf(x), bf(w), b, padding=1)
    assert rel(out[:2], ref) < 1e-4 and rel(out[2:], ref) < 1e-4


def test_per_sample_weights_and_sample_bias():
    from diffusynth_b200 import ops
    N, H, W = 3, 16, 8
    x = cases.randn((N, 128, H, W), 24)
    M = cases.randn((N, 96, 128), 25) * 0.1
    bias, sb = cases.randn((96,), 26), cases.randn((N, 96), 27)
    e2 = torch.zeros(1, 96); e2[0] = bias
    pc = ops.PackedConv(weight=torch.zeros(1, dtype=ops.ACT), e2=e2, e1=None, taps=[[(0, 0, 0)]], cin=128, cout=96, cout_pad=96, ncls=1, kind="s1")
    out = torch.zeros((N, H, W, 96), dtype=ops.ACT, device="cuda")
    _run(pc, [nhwc(x)], N, H, W, out=out, weight_override=M.to(ops.ACT).cuda().contiguous(), per_sample_weights=True, sbias=sb.cuda())
    ref = torch.einsum("nok,nkhw->nohw", bf(M), bf(x)) + bias.view(1, -1, 1, 1) + sb.view(N, -1, 1, 1)
    assert rel(nchw(out), ref) < TOL


def test_invalid_arguments_are_rejected():
    from diffusynth_b200 import _lib, ops
    pc = ops.pack_conv_s1(cases.randn((32, 40, 1, 1), 1), None)     # 40 input channels: not a multiple of 32
    x = torch.zeros((1, 8, 16, 40), dtype=ops.ACT, device="cuda")
    out = torch.zeros((1, 8, 16, 32), dtype=ops.ACT, device="cuda")
    with pytest.raises(_lib.DsError):
        _run(pc, [x], 1, 8, 16, out=out)
