"""ds_conv_gemm and ds_dwconv7 at the scale the benchmark runs them, element by element against the float64 references of
tests/conv_oracle.py.

Both kernels are persistent: a CTA (a CTA pair, a dwconv block) walks a run of work items, and at batch 64 (N = 128 with the
guidance halves) a CTA runs up to ~55 U-Net tiles and a dwconv block up to ~42.  The defects a small test cannot see live there:
the tensor-memory accumulator reused from the third item on (or, with one accumulator per CTA, from the second), the tile decode
at large work indices, the dwconv's second TMA stage and its statistics runs that cross a sample boundary.

(a) The call-site sweep records every convolution of one evaluation of the deployed U-Net at the benchmark's configuration and of
    the VQGAN decoder at batch 64, snapshots each call's inputs (the statistics entry it reads included), launches it and
    compares every output element and the published statistics with the float64 reference of the snapshot.
(b) Synthetic cases reach the rest of the planner's branches at a small cost; each asserts the plan it is meant to run through
    the planner query (ops.conv_plan) or the dwconv grid rule (conv_oracle.dwconv7_grid)."""
import time

import pytest
import torch

from diffusynth_b200 import ops
from oracle import cases
from tests import conv_oracle as CO

pytestmark = pytest.mark.gpu
ACT = ops.ACT
SUBSET_ABOVE = 1 << 21          # pixels x samples above which a call is checked on samples 0, N // 2 and N - 1 only


# ------------------------------------------------------------------------------------------------------------------------------
# one checked call
# ------------------------------------------------------------------------------------------------------------------------------
def _samples(N, H, W):
    return list(range(N)) if N * H * W <= SUBSET_ABOVE else sorted({0, N // 2, N - 1})


def conv_snapshot(pc, src0, src1, N, Hin, Win, kw):
    w = kw.get("weight_override")
    st = kw.get("stats_in")
    return dict(src0=src0.clone(), src1=None if src1 is None else src1.clone(), weight=(pc.weight if w is None else w).clone(),
                mr=None if st is None else st.buf[:, 0].clone(), sbias=None if kw.get("sbias") is None else kw["sbias"].clone(),
                residual=None if kw.get("residual") is None else kw["residual"].clone())


def conv_compare(pc, snap, N, Hin, Win, kw, a, st_out):
    """Worst gate fraction of the outputs of a finished ds_conv_gemm call (16-bit or fp32 output, published statistics)."""
    samples = _samples(N, Hin, Win)
    v, g = CO.conv_gemm_ref(snap["src0"], snap["src1"], snap["weight"], pc.taps, pc.kind, N, Hin, Win, pc.e2, pc.cout, e1=pc.e1,
                            ncls=pc.ncls, mean_rstd=snap["mr"], sbias=snap["sbias"], act=kw.get("act", 0), residual=snap["residual"],
                            src_batch_mod=kw.get("src_batch_mod", 0), per_sample_weights=kw.get("per_sample_weights", False),
                            samples=samples)
    idx = torch.tensor(samples, device=v.device)
    out, out32 = kw.get("out"), kw.get("out_f32")
    res = 0.0
    if out is not None:
        if pc.kind == "up":
            Ho, Wo = 2 * a.H, 2 * a.W
            top, left = (out.shape[1] - Ho) // 2, (out.shape[2] - Wo) // 2
            got = out[idx, top:top + Ho, left:left + Wo, :pc.cout]
            rv, rg = CO.interleave_up(v), CO.interleave_up(g)
        else:
            got, rv, rg = out[idx][..., :pc.cout], v[:, 0], g[:, 0]
        r16, g16 = CO.out16_ref(rv, rg, ACT)
        res = max(res, CO.worst(got, r16, g16))
    if out32 is not None:
        res = max(res, CO.worst(out32[idx].permute(0, 2, 3, 1), v[:, 0], g[:, 0]))
    if st_out is not None:
        assert len(samples) == N
        res = max(res, CO.check_stats(st_out.buf, samples, v, g, st_out.count, a.eps))
    return res


def dw_compare(snap, weight, tbias_stride, out, N, H, W, stats, src_batch_mod, eps):
    samples = _samples(N, H, W)
    v, g = CO.dwconv7_ref(snap["src0"], snap["src1"], weight, snap["tbias"], tbias_stride, N, H, W, src_batch_mod=src_batch_mod,
                          samples=samples)
    r16, g16 = CO.out16_ref(v, g, ACT)
    res = CO.worst(out[torch.tensor(samples, device=out.device)], r16, g16)
    if stats is not None:
        assert len(samples) == N
        res = max(res, CO.check_stats(stats.buf, samples, v, g, H * W * weight.shape[1], eps))
    return res


def _fmt_conv(p):
    return (f"BK {p['BK']:2d} BN {p['BN']:3d} cg {p['cg']} flat {p['pair_flat']} epi {p['epi']} two {p['two_per_sm']} nacc {p['nacc']} "
            f"sps {p['sps']} st {p['stages']} tiles {p['num_tiles']:5d} grid {p['grid']:3d} items/CTA {p['items_per_cta']:6.2f}")


# ------------------------------------------------------------------------------------------------------------------------------
# (a) every call site of the benchmark's U-Net evaluation and VQGAN decode
# ------------------------------------------------------------------------------------------------------------------------------
class Recorder:
    """Wraps a module's conv_args / run_conv and ops.dwconv7: every launch is checked right after it ran, on a snapshot of its inputs."""

    def __init__(self, monkeypatch, mod):
        self.rows, self.name, self.calls = [], "", {}
        orig_args, orig_run, orig_dw = mod.conv_args, mod.run_conv, ops.dwconv7

        def conv_args(pc, src0, src1, N, Hin, Win, **kw):
            a, st, keep = orig_args(pc, src0, src1, N, Hin, Win, **kw)
            self.calls[id(a)] = (pc, src0, src1, N, Hin, Win, kw, a, st)
            return a, st, keep

        def run_conv(a, reference=False):
            pc, src0, src1, N, Hin, Win, kw, a_, st = self.calls[id(a)]
            assert a_ is a and not reference
            plan = ops.conv_plan(a)
            snap = conv_snapshot(pc, src0, src1, N, Hin, Win, kw)
            orig_run(a)
            torch.cuda.synchronize()
            w = conv_compare(pc, snap, N, Hin, Win, kw, a, st)
            self.rows.append(("conv", self.name, plan, w))

        def dwconv7(src0, src1, weight, tbias, tbias_stride, out, N, H, W, stats=None, src_batch_mod=0, eps=1e-5):
            snap = dict(src0=src0.clone(), src1=None if src1 is None else src1.clone(), tbias=tbias.clone())
            orig_dw(src0, src1, weight, tbias, tbias_stride, out, N, H, W, stats=stats, src_batch_mod=src_batch_mod, eps=eps)
            torch.cuda.synchronize()
            w = dw_compare(snap, weight, tbias_stride, out, N, H, W, stats, src_batch_mod, eps)
            grid = CO.dwconv7_grid(weight.shape[1], H, W, N, torch.cuda.get_device_properties(0).multi_processor_count)
            self.rows.append(("dw", self.name, grid, w))

        monkeypatch.setattr(mod, "conv_args", conv_args)
        monkeypatch.setattr(mod, "run_conv", run_conv)
        monkeypatch.setattr(ops, "dwconv7", dwconv7)

    def run(self, plan_ops):
        for name, fn in plan_ops:
            self.name = name
            fn()


def test_call_sites_of_the_benchmark_evaluation(monkeypatch):
    from diffusynth_b200 import VQGAN, ConditionedUnet, unet as unet_mod, vqgan as vqgan_mod, weights as W
    t0 = time.time()
    g = torch.Generator().manual_seed(17)
    # the deployed U-Net as the sampling loop runs it at batch 64: N = 128 (both guidance halves), one timestep for the batch, the
    # prefix up to downs.0.0 evaluated once for the 64 distinct latents
    rec = Recorder(monkeypatch, unet_mod)
    net = ConditionedUnet(**{k: v for k, v in W.UNET_DEPLOYED.items() if k not in ("out_dim", "time_dim")}, device="cuda")
    net.load_state_dict(W.unet_random_state_dict(seed=3))
    net.use_engine = False
    pl = net.plan(128, 128, 64, x_batch_mod=64, uniform_time=True)
    assert pl.shared == 64
    pl.x.copy_(torch.randn(pl.x.shape, generator=g))
    pl.t.fill_(421)
    pl.cond.copy_(torch.randn(pl.cond.shape, generator=g).to(pl.cond.dtype))
    pl.run_cond()
    rec.run(pl.ops)
    unet_rows = rec.rows
    # the VQGAN decoder on quantised latents of a batch of 64
    rec = Recorder(monkeypatch, vqgan_mod)
    vq = VQGAN(**W.VQGAN_DEPLOYED, device="cuda")
    vq.load_state_dict(W.vqgan_random_state_dict(seed=4))
    q, _, _ = vq._vq_vae(torch.randn((64, 4, 128, 64), generator=g).cuda())
    dpl = vq._decoder._stack.plan(64, 128, 64)
    dpl.inp.copy_(q)
    rec.run(dpl.ops)
    rows = unet_rows + rec.rows
    torch.cuda.synchronize()

    print(f"\n{len(rows)} calls checked in {time.time() - t0:.1f} s; worst error as a fraction of its gate:")
    for kind, name, p, w in rows:
        desc = _fmt_conv(p) if kind == "conv" else (f"dwconv {p['kernel']} tiles {p['tiles']:3d} grid {p['grid']:5d} "
                                                      f"items/block {p['per_block']:3d} crosses sample {int(p['crosses_sample'])}")
        print(f"  {name:34s} {desc}  worst {w:.3f}")
    bad = [(name, w) for _, name, _, w in rows if not w <= 1.0]
    assert not bad, bad
    convs = [p for kind, _, p, _ in rows if kind == "conv"]
    dws = [p for kind, _, p, _ in rows if kind == "dw"]
    assert sum(kind == "conv" for kind, _, _, _ in unet_rows) == 82 and len(dws) == 22 and len(convs) > 82
    assert {p["cg"] for p in convs} == {1, 2} and any(p["pair_flat"] for p in convs)
    assert {p["nacc"] for p in convs if p["two_per_sm"]} == {1, 2}
    assert {192, 256} <= {p["BN"] for p in convs}
    # every epilogue these models run (epilogue 1, the fold without GELU, runs only with the unfused attention's to_qkv: the
    # synthetic 1x1 cases below cover it)
    assert {p["epi"] for p in convs} == {0, 2, 3, 4}
    assert max(p["items_per_cta"] for p in convs) >= 3
    assert any(p["items_per_cta"] >= 3 for p in convs if p["cg"] == 2)
    assert any(p["kernel"] == "mma" and p["per_block"] > 1 and p["crosses_sample"] for p in dws)


# ------------------------------------------------------------------------------------------------------------------------------
# the float64 reference on the device
# ------------------------------------------------------------------------------------------------------------------------------
def test_device_reference_equals_the_cpu_reference():
    x0, x1 = cases.randn((2, 64, 12, 9), 1).permute(0, 2, 3, 1).to(ACT), cases.randn((4, 32, 12, 9), 2).permute(0, 2, 3, 1).to(ACT)
    pc = ops.pack_conv_s1(cases.randn((40, 96, 3, 3), 3) * 0.1, cases.randn((40,), 4), 1 + 0.1 * cases.randn((96,), 5), cases.randn((96,), 6))
    mr = torch.tensor([[0.3, 1.7], [-0.2, 0.9]])
    sb = cases.randn((4, 48), 7)
    kw = dict(e1=pc.e1, ncls=pc.ncls, mean_rstd=mr, sbias=sb, act=1, src_batch_mod=2)
    vc, gc = CO.conv_gemm_ref(x0, x1, pc.weight, pc.taps, "s1", 4, 12, 9, pc.e2, pc.cout, **kw)
    dev = {k: (t.cuda() if isinstance(t, torch.Tensor) else t) for k, t in kw.items()}
    vd, gd = CO.conv_gemm_ref(x0.cuda(), x1.cuda(), pc.weight.cuda(), pc.taps, "s1", 4, 12, 9, pc.e2.cuda(), pc.cout, **dev)
    assert torch.allclose(vd.cpu(), vc, rtol=1e-12, atol=1e-12) and torch.allclose(gd.cpu(), gc, rtol=1e-9)
    wt, tb = cases.randn((49, 96), 8) * 0.1, cases.randn((4, 96), 9)
    for H in (16, 12):
        xs = cases.randn((4, 96, H, 9), 10).permute(0, 2, 3, 1).to(ACT)
        vc, gc = CO.dwconv7_ref(xs, None, wt, tb, 96, 4, H, 9)
        vd, gd = CO.dwconv7_ref(xs.cuda(), None, wt.cuda(), tb.cuda(), 96, 4, H, 9)
        assert torch.allclose(vd.cpu(), vc, rtol=1e-12, atol=1e-12) and torch.allclose(gd.cpu(), gc, rtol=1e-9)


# ------------------------------------------------------------------------------------------------------------------------------
# (b) synthetic cases
# ------------------------------------------------------------------------------------------------------------------------------
def build_conv_case(spec, device="cuda", seed=0):
    """One ds_conv_gemm call from a case spec; returns (pc, src0, src1, N, Hin, Win, kw, a, stats_out)."""
    kind, cin, c1, cout, k, H, W, N = (spec[f] for f in ("kind", "cin", "c1", "cout", "k", "H", "W", "N"))
    opt = spec.get
    mod = opt("mod", 0)
    n0 = mod if mod else N
    x0 = (cases.randn((n0, H, W, cin), seed + 1) + opt("shift", 0.0)).to(ACT).to(device)
    x1 = cases.randn((N, H, W, c1), seed + 2).to(ACT).to(device) if c1 else None
    fold = opt("fold", False)
    if kind == "down":
        pc = ops.pack_conv_down(cases.randn((cout, cin, 4, 4), seed + 3) * (cin * 16) ** -0.5, cases.randn((cout,), seed + 4))
    elif kind == "up":
        pc = ops.pack_conv_up(cases.randn((cin, cout, 4, 4), seed + 3) * (cin * 4) ** -0.5, cases.randn((cout,), seed + 4))
    elif opt("per_sample"):
        e2 = torch.zeros(1, ops.pad16(cout)); e2[0, :cout] = cases.randn((cout,), seed + 4)
        pc = ops.PackedConv(weight=torch.zeros(1, dtype=ACT), e2=e2, e1=None, taps=[[(0, 0, 0)]], cin=cin, cout=cout,
                            cout_pad=ops.pad16(cout), ncls=1, kind="s1")
    else:
        ct = cin + c1
        gamma, beta = (1 + 0.2 * cases.randn((ct,), seed + 5), 0.3 * cases.randn((ct,), seed + 6)) if fold else (None, None)
        pc = ops.pack_conv_s1(cases.randn((cout, ct, k, k), seed + 3) * (ct * k * k) ** -0.5, cases.randn((cout,), seed + 4), gamma, beta)
    pc.to(device)
    kw = dict(act=opt("act", 0), src_batch_mod=mod)
    Ho, Wo = (H // 2, W // 2) if kind == "down" else (2 * H, 2 * W) if kind == "up" else (H, W)
    if fold:
        xb = torch.cat([x0[torch.arange(N, device=device) % n0] if mod else x0] + ([x1] if c1 else []), -1).double()
        mean = xb.mean(dim=(1, 2, 3))[:n0]
        rstd = (xb.var(dim=(1, 2, 3), unbiased=False) + 1e-5).rsqrt()[:n0]
        kw["stats_in"] = ops.given_stats(mean.float().cpu(), rstd.float().cpu(), xb[0].numel(), device)
    if opt("sbias"):
        kw["sbias"] = cases.randn((N, pc.cout_pad + 3), seed + 7).to(device)
    if opt("residual"):
        kw["residual"] = cases.randn((N, Ho, Wo, cout), seed + 8).to(ACT).to(device)
    if opt("per_sample"):
        kw["weight_override"] = (cases.randn((N, pc.cout_pad, cin), seed + 9) * cin ** -0.5).to(ACT).to(device)
        kw["per_sample_weights"] = True
    if opt("out_f32"):
        kw["out_f32"] = torch.full((N, cout, Ho, Wo), float("nan"), device=device)
    else:
        pad = opt("pad_up", 0)
        kw["out"] = torch.zeros((N, Ho + pad, Wo + pad, cout), dtype=ACT, device=device)
    a, st, _ = ops.conv_args(pc, x0, x1, N, H, W, want_stats=opt("stats", False), **kw)
    return pc, x0, x1, N, H, W, kw, a, st


CONV_CASES = {
    # cg = 1: >= 3 items per CTA at BK 32 / 64 and BN 96 / 192 / 256 (GroupNorm fold: one CTA per SM)
    "1x1_bk32_bn96": (dict(kind="s1", cin=96, c1=0, cout=96, k=1, H=32, W=16, N=128, fold=True, shift=0.5, stats=True),
                      dict(BK=32, BN=96, cg=1, epi=1, two_per_sm=0)),
    "1x1_bk64_bn192": (dict(kind="s1", cin=384, c1=0, cout=384, k=1, H=16, W=8, N=512, fold=True, sbias=True),
                       dict(BK=64, BN=192, cg=1, epi=1, two_per_sm=0)),
    "1x1_bk64_bn256": (dict(kind="s1", cin=256, c1=0, cout=768, k=1, H=16, W=8, N=256, fold=True),
                       dict(BK=64, BN=256, cg=1, epi=1)),
    # two CTAs per SM: one tensor-memory accumulator per CTA (BN = 192) and two (BN = 96)
    "1x1_two_per_sm_nacc1": (dict(kind="s1", cin=384, c1=0, cout=384, k=1, H=16, W=16, N=256),
                             dict(BN=192, cg=1, epi=4, two_per_sm=1, nacc=1)),
    "1x1_two_per_sm_nacc2": (dict(kind="s1", cin=96, c1=0, cout=96, k=1, H=64, W=32, N=128),
                             dict(BN=96, cg=1, epi=4, two_per_sm=1, nacc=2)),
    # cg = 2 pairs
    "3x3_cg2_bk32_bn96_gelu": (dict(kind="s1", cin=96, c1=0, cout=96, k=3, H=32, W=32, N=64, fold=True, act=1, stats=True),
                               dict(BK=32, BN=96, cg=2, pair_flat=0, epi=2)),
    "3x3_cg2_flat_bk64_bn192_res": (dict(kind="s1", cin=192, c1=0, cout=384, k=3, H=16, W=8, N=256, fold=True, residual=True, stats=True),
                                    dict(BK=64, BN=192, cg=2, pair_flat=1, epi=3)),
    "3x3_cg2_flat_bn256": (dict(kind="s1", cin=256, c1=0, cout=512, k=3, H=16, W=8, N=256),
                           dict(BK=64, BN=256, cg=2, pair_flat=1, epi=4)),
    "3x3_two_sources_batch_mod": (dict(kind="s1", cin=96, c1=192, cout=192, k=3, H=32, W=16, N=128, mod=64, fold=True, act=1, stats=True),
                                  dict(BK=32, BN=192, cg=2, epi=2)),
    # ragged maps: partial tiles in both directions on late items
    "3x3_ragged": (dict(kind="s1", cin=64, c1=0, cout=64, k=3, H=20, W=12, N=160, fold=True, residual=True, stats=True),
                   dict(BK=64, cg=2, epi=3)),
    "3x3_ragged_odd_tiles": (dict(kind="s1", cin=64, c1=0, cout=128, k=3, H=24, W=20, N=127, fold=True, act=1),
                             dict(cg=1, epi=2)),
    # stride-2 down with odd sizes and the transposed conv into a padded map, at large N
    "down_odd": (dict(kind="down", cin=96, c1=0, cout=192, k=4, H=65, W=33, N=128), dict(cg=2, epi=4)),
    "up_padded": (dict(kind="up", cin=192, c1=0, cout=96, k=4, H=16, W=12, N=128, pad_up=1), dict(cg=2, epi=4)),
    # attention to_out: per-sample weights, with and without a per-sample bias
    "per_sample_weights": (dict(kind="s1", cin=128, c1=0, cout=96, k=1, H=32, W=16, N=128, per_sample=True, stats=True),
                           dict(cg=1, epi=4)),
    "per_sample_weights_sbias": (dict(kind="s1", cin=128, c1=0, cout=96, k=1, H=32, W=16, N=128, per_sample=True, sbias=True),
                                 dict(cg=1, epi=1)),
    # final conv: fp32 NCHW output of 4 real channels, source 0 shared by the guidance halves
    "final_fp32_nchw_batch_mod": (dict(kind="s1", cin=96, c1=0, cout=4, k=3, H=128, W=64, N=128, mod=64, out_f32=True), dict(epi=0)),
}


@pytest.mark.parametrize("case", sorted(CONV_CASES))
def test_conv_gemm_synthetic(case):
    spec, want = CONV_CASES[case]
    pc, x0, x1, N, H, W, kw, a, st = build_conv_case(spec)
    plan = ops.conv_plan(a)
    print(f"\n{case}: {_fmt_conv(plan)}")
    assert {k: plan[k] for k in want} == want
    assert plan["items_per_cta"] >= (1 if plan["two_per_sm"] else 3)
    snap = conv_snapshot(pc, x0, x1, N, H, W, kw)
    ops.run_conv(a)
    torch.cuda.synchronize()
    w = conv_compare(pc, snap, N, H, W, kw, a, st)
    print(f"{case}: worst {w:.3f}")
    assert w <= 1.0
    if st is not None:        # a second launch into the same statistics buffer publishes the same bits
        first = st.buf.clone()
        ops.run_conv(a)
        torch.cuda.synchronize()
        assert torch.equal(first, st.buf)
    if spec.get("pad_up"):
        out = kw["out"]
        assert float(out[:, -1].abs().max()) == 0.0 and float(out[:, :, -1].abs().max()) == 0.0


DW_CASES = {
    # >= 3 items per block at the U-Net widths and the concatenations of the up path (a run crosses a sample boundary)
    "c96": dict(C0=96, C1=0, H=32, W=16, N=160),
    "c192": dict(C0=192, C1=0, H=32, W=16, N=96),
    "c384": dict(C0=384, C1=0, H=16, W=16, N=96),
    "c768": dict(C0=768, C1=0, H=16, W=8, N=64),
    "c288_concat": dict(C0=96, C1=192, H=32, W=32, N=40),
    "c576_concat": dict(C0=192, C1=384, H=16, W=24, N=48),
    # source 0 shared by the two guidance halves, with a second source; one bias row for every sample
    "batch_mod_two_sources": dict(C0=96, C1=192, H=32, W=16, N=64, mod=32),
    "tbias_stride0": dict(C0=192, C1=0, H=32, W=16, N=64, stride0=True),
    # the FFMA2 kernel (maps shorter than 16 rows)
    "ffma2_h8": dict(C0=96, C1=0, H=8, W=8, N=6),
    "ffma2_h12": dict(C0=192, C1=96, H=12, W=13, N=5, mod=3),
    "ffma2_h15": dict(C0=384, C1=0, H=15, W=7, N=4, stride0=True),
    # 16-row tiles with a partial last tile, and the odd widths of note synthesis
    "h16_w3": dict(C0=96, C1=0, H=16, W=3, N=200),
    "h17_w7": dict(C0=192, C1=0, H=17, W=7, N=100),
    "h20_w15": dict(C0=96, C1=96, H=20, W=15, N=90),
}


@pytest.mark.parametrize("case", sorted(DW_CASES))
def test_dwconv7_synthetic(case):
    c = DW_CASES[case]
    C0, C1, H, W, N, mod = c["C0"], c["C1"], c["H"], c["W"], c["N"], c.get("mod", 0)
    C = C0 + C1
    grid = CO.dwconv7_grid(C, H, W, N, torch.cuda.get_device_properties(0).multi_processor_count)
    print(f"\n{case}: {grid}")
    if H >= 16 and not case.startswith("h"):
        assert grid["kernel"] == "mma" and grid["per_block"] >= 3 and grid["crosses_sample"]
    assert grid["kernel"] == ("ffma2" if H < 16 else "mma")
    src0 = (cases.randn((mod or N, H, W, C0), 1) + 0.3).to(ACT).cuda()
    src1 = cases.randn((N, H, W, C1), 2).to(ACT).cuda() if C1 else None
    weight = (cases.randn((49, C), 3) * 0.15).cuda()
    tbias = cases.randn((1, C) if c.get("stride0") else (N, C + 5), 4).cuda()
    stride = 0 if c.get("stride0") else tbias.shape[1]
    out = torch.full((N, H, W, C), float("nan"), dtype=ACT, device="cuda")
    st = ops.dwconv7_stats(N, C, H, W, "cuda")
    snap = dict(src0=src0.clone(), src1=None if src1 is None else src1.clone(), tbias=tbias.clone())
    ops.dwconv7(src0, src1, weight, tbias, stride, out, N, H, W, stats=st, src_batch_mod=mod)
    torch.cuda.synchronize()
    w = dw_compare(snap, weight, stride, out, N, H, W, st, mod, 1e-5)
    print(f"{case}: worst {w:.3f}")
    assert w <= 1.0
    first = st.buf.clone()
    ops.dwconv7(src0, src1, weight, tbias, stride, out, N, H, W, stats=st, src_batch_mod=mod)
    torch.cuda.synchronize()
    assert torch.equal(first, st.buf)
