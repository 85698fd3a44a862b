"""The float64 convolution references of tests/conv_oracle.py, without a GPU: pinned to F.conv2d / F.conv_transpose2d in float64 and
to the fp32 contract() of tests/test_host_packing.py, and each gate shown to be tight -- a reference that is wrong in one K-block
of one tile, one tile, one border row, the dwconv weight rounding or one statistics slot misses its gate by 10x or more.  Also
pins a few launch plans of the ds_conv_gemm planner query (no device: 148 SMs)."""
import pytest
import torch
import torch.nn.functional as F

from diffusynth_b200 import ops
from oracle import cases
from tests import conv_oracle as CO
from tests.test_host_packing import contract

ACT = ops.ACT
MARGIN = 10.0


def act16(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous().to(ACT)


def ref(pc, srcs, N, Hin, Win, **kw):
    return CO.conv_gemm_ref(srcs[0], srcs[1] if len(srcs) > 1 else None, pc.weight, pc.taps, pc.kind, N, Hin, Win, pc.e2, pc.cout,
                            e1=pc.e1, ncls=pc.ncls, **kw)


def nchw64(x):
    return x.double().permute(0, 3, 1, 2)


@pytest.mark.parametrize("k", [1, 3])
def test_s1_two_sources_and_batch_mod_match_conv2d(k):
    N, mod = 4, 2
    x0, x1 = cases.randn((mod, 64, 9, 12), 1), cases.randn((N, 32, 9, 12), 2)
    w, b = cases.randn((48, 96, k, k), 3) * 0.1, cases.randn((48,), 4)
    pc = ops.pack_conv_s1(w, b)
    v, g = ref(pc, [act16(x0), act16(x1)], N, 9, 12, src_batch_mod=mod)
    xin = torch.cat([act16(x0)[torch.arange(N) % mod], act16(x1)], dim=-1)
    want = F.conv2d(nchw64(xin), w.to(ACT).double(), b.double(), padding=k // 2)
    assert torch.allclose(nchw64(v[:, 0]), want, rtol=1e-12, atol=1e-12)
    assert bool((g > 0).all())


@pytest.mark.parametrize("H,W", [(16, 12), (9, 7), (32, 13)])
def test_down_and_up_match_torch(H, W):
    N = 2
    x = cases.randn((N, 32, H, W), 5)
    w, b = cases.randn((48, 32, 4, 4), 6) * 0.1, cases.randn((48,), 7)
    pc = ops.pack_conv_down(w, b)
    v, _ = ref(pc, [act16(x)], N, H, W)
    want = F.conv2d(nchw64(act16(x)), w.to(ACT).double(), b.double(), stride=2, padding=1)
    assert torch.allclose(nchw64(v[:, 0]), want, rtol=1e-12, atol=1e-12)
    wt, bt = cases.randn((32, 48, 4, 4), 8) * 0.1, cases.randn((48,), 9)
    pcu = ops.pack_conv_up(wt, bt)
    vu, _ = ref(pcu, [act16(x)], N, H, W)
    want = F.conv_transpose2d(nchw64(act16(x)), wt.to(ACT).double(), bt.double(), stride=2, padding=1)
    assert torch.allclose(nchw64(CO.interleave_up(vu)), want, rtol=1e-12, atol=1e-12)


def _fold_case(seed=10, N=2, H=16, W=24, act=1):
    x = cases.randn((N, 96, H, W), seed) * 1.5 + 0.8
    w, b = cases.randn((64, 96, 3, 3), seed + 1) * 0.05, cases.randn((64,), seed + 2)
    gamma, beta = 1 + 0.2 * cases.randn((96,), seed + 3), 0.5 * cases.randn((96,), seed + 4)
    pc = ops.pack_conv_s1(w, b, gamma, beta)
    xs = act16(x)
    xb = xs.double()
    mean = xb.mean(dim=(1, 2, 3))
    rstd = (xb.var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt()
    mr = torch.stack([mean, rstd], 1).float()
    sb = cases.randn((N, 64), seed + 5)
    res = act16(cases.randn((N, 64, H, W), seed + 6))
    return pc, xs, mr, sb, res


def test_fold_gelu_residual_agrees_with_fp32_contract_within_the_gates():
    pc, xs, mr, _, res = _fold_case()
    N, H, W = xs.shape[0], xs.shape[1], xs.shape[2]
    for act, resid in ((1, None), (0, res)):
        v, g = ref(pc, [xs], N, H, W, mean_rstd=mr, act=act, residual=resid)
        for n in range(N):
            c = contract(pc, [xs[n:n + 1].float().permute(0, 3, 1, 2)], "s1", (mr[n, 0], mr[n, 1]), act=act,
                         residual=None if resid is None else resid[n:n + 1].float().permute(0, 3, 1, 2))
            assert CO.worst(c.permute(0, 2, 3, 1), v[n:n + 1, 0], g[n:n + 1, 0]) <= 1.0


def test_dwconv_matches_depthwise_conv2d_with_the_kernel_weights():
    N, C = 3, 64
    for H, W in ((16, 8), (12, 7)):
        x0, x1 = cases.randn((2, 32, H, W), 11), cases.randn((N, 32, H, W), 12)
        wt = cases.randn((49, C), 13) * 0.1
        tb = cases.randn((N, C + 8), 14)
        v, g = CO.dwconv7_ref(act16(x0), act16(x1), wt, tb, tb.shape[1], N, H, W, src_batch_mod=2)
        wk = (wt.to(ACT) if H >= 16 else wt).double().t().reshape(C, 1, 7, 7)
        xin = torch.cat([act16(x0)[torch.arange(N) % 2], act16(x1)], -1)
        want = F.conv2d(nchw64(xin), wk, None, padding=3, groups=C) + tb[:, :C].double().view(N, C, 1, 1)
        assert torch.allclose(nchw64(v), want, rtol=1e-12, atol=1e-12)
        v0, _ = CO.dwconv7_ref(act16(x0), act16(x1), wt, tb[0], 0, N, H, W, src_batch_mod=2)     # one bias row for every sample
        want0 = want - tb[:, :C].double().view(N, C, 1, 1) + tb[0, :C].double().view(1, C, 1, 1)
        assert torch.allclose(nchw64(v0), want0, rtol=1e-12, atol=1e-12)


def test_stats_reference():
    v = cases.randn((3, 5, 7, 16), 15).double() * 2 + 0.3
    g = torch.full_like(v, 1e-6)
    (s, q, m, r), gates = CO.stats_ref(v, g, 5 * 7 * 16, 1e-5)
    assert torch.allclose(m, v.mean(dim=(1, 2, 3))) and torch.allclose(s, v.sum(dim=(1, 2, 3)))
    assert torch.allclose(r, (v.var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt())
    assert all(bool((t > 0).all()) for t in gates)


# ---- the gates are tight: each defect a kernel could have moves its metric by >= 10x the gate ----------------------------------
def _out(v, g):
    return CO.out16_ref(v, g, ACT)


def test_gate_catches_one_dropped_k_block_in_one_tile():
    pc, xs, mr, _, _ = _fold_case(act=0)
    N, H, W = xs.shape[0], xs.shape[1], xs.shape[2]
    v, g = ref(pc, [xs], N, H, W, mean_rstd=mr)
    r, gr = _out(v, g)
    wm = pc.weight.clone()
    wm[0, :, 4 * 96 + 32:4 * 96 + 64] = 0            # K-block (BK = 32) 1 of the centre tap
    pm = ops.PackedConv(weight=wm, e2=pc.e2, e1=pc.e1, taps=pc.taps, cin=pc.cin, cout=pc.cout, cout_pad=pc.cout_pad, ncls=9, kind="s1")
    vm, _ = ref(pm, [xs], N, H, W, mean_rstd=mr)
    hb, wb = ops.choose_tile(H, W)
    bad = v.clone()
    bad[1, 0, :hb, wb:2 * wb, :32] = vm[1, 0, :hb, wb:2 * wb, :32]     # one M-tile x one 32-column N-tile
    assert not torch.equal(bad, v)
    assert CO.worst(r, r, gr) == 0.0
    assert CO.worst(bad, r, gr) >= MARGIN


def test_gate_catches_a_tile_from_the_wrong_sample_and_a_stale_accumulator():
    pc = ops.pack_conv_s1(cases.randn((32, 64, 3, 3), 20) * 0.05, cases.randn((32,), 21))
    N, H, W = 2, 32, 16
    xs = act16(cases.randn((N, 64, H, W), 22))
    v, g = ref(pc, [xs], N, H, W)
    r, gr = _out(v, g)
    hb, wb = ops.choose_tile(H, W)
    t0, t1 = (slice(0, hb), slice(0, wb)), (slice(hb, 2 * hb), slice(0, wb))
    wrong = v.clone()
    wrong[1, 0, t0[0], t0[1]] = v[0, 0, t0[0], t0[1]]
    assert CO.worst(wrong, r, gr) >= MARGIN
    e2c = pc.e2[0, :32].double()
    stale = v.clone()
    stale[0, 0, t1[0], t1[1]] += v[0, 0, t0[0], t0[1]] - e2c        # accumulator of the previous item not cleared
    assert CO.worst(stale, r, gr) >= MARGIN


def test_gate_catches_a_wrong_border_class_on_the_last_row():
    pc, xs, mr, _, _ = _fold_case(act=0)
    N, H, W = xs.shape[0], xs.shape[1], xs.shape[2]
    v, g = ref(pc, [xs], N, H, W, mean_rstd=mr)
    r, gr = _out(v, g)
    e1m, e2m = pc.e1.clone(), pc.e2.clone()
    e1m[6:9], e2m[6:9] = pc.e1[3:6], pc.e2[3:6]             # bottom row evaluated with the middle rows' tables
    pm = ops.PackedConv(weight=pc.weight, e2=e2m, e1=e1m, taps=pc.taps, cin=pc.cin, cout=pc.cout, cout_pad=pc.cout_pad, ncls=9, kind="s1")
    vm, _ = ref(pm, [xs], N, H, W, mean_rstd=mr)
    assert torch.equal(vm[:, :, :-1], v[:, :, :-1])
    assert CO.worst(vm, r, gr) >= MARGIN


def test_gate_catches_unrounded_weights_in_the_tensor_core_dwconv():
    N, C, H, W = 2, 96, 16, 24
    xs = act16(cases.randn((N, C, H, W), 30))
    wt = cases.randn((49, C), 31) * 0.1
    tb = cases.randn((N, C), 32)
    v, g = CO.dwconv7_ref(xs, None, wt, tb, C, N, H, W)
    r, gr = _out(v, g)
    xin = nchw64(xs)
    unrounded = F.conv2d(xin, wt.double().t().reshape(C, 1, 7, 7), None, padding=3, groups=C) + tb.double().view(N, C, 1, 1)
    assert CO.worst(unrounded.permute(0, 2, 3, 1), r, gr) >= MARGIN


def test_gate_catches_one_missing_stats_slot():
    N, C, H, W = 2, 64, 32, 16
    xs = act16(cases.randn((N, C, H, W), 40) + 0.5)
    wt = cases.randn((49, C), 41) * 0.1
    tb = cases.randn((N, C), 42)
    v, g = CO.dwconv7_ref(xs, None, wt, tb, C, N, H, W)
    (s, q, m, r), (gs, gq, gm, gr) = CO.stats_ref(v, g, H * W * C, 1e-5)
    tile = v[:, :16, :16, :32]                      # one (16 x 16 pixels, 32 channels) slot of the tensor-core kernel
    assert CO.worst(s - tile.sum(dim=(1, 2, 3)), s, gs) >= MARGIN
    assert CO.worst(q - (tile * tile).sum(dim=(1, 2, 3)), q, gq) >= MARGIN


# ---- planner query ---------------------------------------------------------------------------------------------------------------
def _plan(cin, cout, k, H, W, N, **kw):
    pc = ops.pack_conv_s1(torch.zeros(cout, cin, k, k), torch.zeros(cout))
    x = torch.zeros((N, H, W, cin), dtype=ACT)
    out = torch.zeros((N, H, W, cout), dtype=ACT)
    a, _, _ = ops.conv_args(pc, x, None, N, H, W, out=out, **kw)
    return ops.conv_plan(a)


def test_planner_query_known_plans():
    """With no device the library plans for 148 SMs (a B200)."""
    p = _plan(96, 96, 3, 128, 64, 128)          # level-0 3x3 of the batch-64 U-Net evaluation: 55 pairs of M-tiles per CTA pair
    assert (p["BK"], p["BN"], p["cg"], p["pair_flat"], p["epi"], p["num_tiles"], p["grid"]) == (32, 96, 2, 0, 4, 4096, 148)
    p = _plan(384, 384, 1, 16, 8, 128)          # deepest level 1x1: two CTAs per SM, one accumulator each (BN = 192)
    assert (p["BN"], p["cg"], p["two_per_sm"], p["nacc"], p["num_tiles"], p["grid"]) == (192, 1, 1, 1, 256, 256)
    p = _plan(64, 64, 3, 16, 8, 2)              # one M-tile per sample: the pair spans two samples
    assert (p["BN"], p["cg"], p["pair_flat"], p["grid"]) == (32, 2, 1, 4)
    p = _plan(64, 768, 1, 16, 8, 2)             # a small job takes narrow N tiles
    assert (p["BN"], p["two_per_sm"], p["nacc"], p["num_tiles"], p["grid"]) == (64, 1, 2, 24, 24)
    p = _plan(128, 96, 3, 16, 24, 3)            # three M-tiles per sample, odd sample count: one CTA per M-tile
    assert (p["cg"], p["pair_flat"]) == (1, 0)
    assert p["items_per_cta"] == p["num_tiles"] / p["grid"]


def test_dwconv_grid_rule():
    g = CO.dwconv7_grid(96, 128, 64, 128)
    assert (g["kernel"], g["tiles"], g["grid"], g["per_block"], g["crosses_sample"]) == ("mma", 32, 98, 42, True)
    g = CO.dwconv7_grid(768, 16, 8, 128)
    assert (g["grid"], g["per_block"]) == (12, 11)
    assert CO.dwconv7_grid(96, 12, 8, 4)["kernel"] == "ffma2"
