"""Time timbre morphs on the GPU (deployed architecture, random-init weights, 20 DDIM steps, CFG 6, w = 64):
  (a) TextToTimbre.morph of P = 8 sequences x N = 16 frames as one launch of 128 rows, against the same 8 sequences as 8 separate
      16-row morph calls (alternated);
  (b) TextToTimbre.invert at B = 64;
  (c) ds_morph_rows alone at P = 64, N = 16, both paths, against the HBM bound of the bytes it must move (endpoints read once,
      rows written once) at the 7.7 TB/s data-sheet figure; the rows written (136 MB) exceed the 126 MB L2.  The time is per
      codec.morph_rows call, events around the call: it includes the wrapper's output allocation, so it bounds the kernels from above.
Prints one JSON line (and writes it to --out): the card, its power limit and maximum SM clock read in the same run, and the
device-timed medians (CUDA events around each call, after a warm-up) of --repeats calls.  Exits non-zero without a CUDA device.

    python tools_dev/morph_time.py --out profiles/morph_time.json"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools_dev"))

from inpaint_time import card  # noqa: E402

HBM_TBPS = 7.7


def timed(fn, repeats):
    import numpy as np
    import torch
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), [round(min(ms), 4), round(max(ms), 4)]


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("morph_time: needs a CUDA device", file=sys.stderr)
        return 2
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases

    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    P, N, L = 8, 16, 512
    e0, e1 = cases.randn((P, 4, 128, 64), 1).cuda(), cases.randn((P, 4, 128, 64), 2).cuda()
    c0, c1 = cases.randn((P, L), 3).cuda(), cases.randn((P, L), 4).cuda()
    _, uncond = W.synthetic_conditions(1, L)
    uncond = uncond.cuda()

    def batched():
        pipe.morph(e0, e1, c0, c1, uncond, N, steps=a.steps, seed=0)

    def per_sequence():
        for p in range(P):
            pipe.morph(e0[p], e1[p], c0[p], c1[p], uncond, N, steps=a.steps, seed=0)

    batched()
    per_sequence()
    torch.cuda.synchronize()
    ms = {"batched": [], "per_sequence": []}
    launches = {}
    for _ in range(a.repeats):
        for k, fn in (("batched", batched), ("per_sequence", per_sequence)):       # alternate the two
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            fn()
            t1.record()
            t1.synchronize()
            ms[k].append(t0.elapsed_time(t1))
            launches[k] = pipe.last_launches * (1 if k == "batched" else P)
    med = {k: float(np.median(v)) for k, v in ms.items()}

    Bi = 64
    lat = cases.vq_latents(B=Bi, seed=5).cuda()
    icond, _ = W.synthetic_conditions(Bi, L)
    icond = icond.cuda()
    inv_ms, inv_mm = timed(lambda: pipe.invert(lat, icond, steps=a.steps), a.repeats)
    inv_launches = pipe.last_launches

    Pk = 64
    k0, k1 = torch.randn((Pk, 4 * 128 * 64), device="cuda"), torch.randn((Pk, 4 * 128 * 64), device="cuda")
    kc0, kc1 = torch.randn((Pk, L), device="cuda"), torch.randn((Pk, L), device="cuda")
    n = 4 * 128 * 64
    kernel = {}
    for path in ("linear", "slerp"):
        t, mm = timed(lambda: codec.morph_rows(k0, k1, kc0, kc1, N, path), max(a.repeats, 50))
        # endpoints read once (both paths; slerp's reduction reads them a second time, counted), rows written once
        reads = 2 * Pk * (n + L) * 4 * (2 if path == "slerp" else 1)
        nbytes = reads + Pk * N * (n + L) * 4
        bound_ms = nbytes / (HBM_TBPS * 1e12) * 1e3
        kernel[path] = dict(ms=round(t, 4), ms_min_max=mm, bytes=nbytes, hbm_bound_ms=round(bound_ms, 4),
                            share_of_hbm_bound=round(bound_ms / t, 3), tb_per_s=round(nbytes / (t * 1e-3) / 1e12, 3))

    name, power, clk = card()
    line = dict(tool="morph_time", card=name, power_limit=power, max_sm_clock=clk, steps=a.steps, cfg_scale=6, width=64, sampler="ddim",
                repeats=a.repeats, weights="deployed architecture, random init",
                morph_sequences=P, morph_frames=N, morph_batched_ms=round(med["batched"], 3),
                morph_batched_ms_min_max=[round(min(ms["batched"]), 3), round(max(ms["batched"]), 3)],
                morph_per_sequence_ms=round(med["per_sequence"], 3),
                morph_per_sequence_ms_min_max=[round(min(ms["per_sequence"]), 3), round(max(ms["per_sequence"]), 3)],
                batched_speedup=round(med["per_sequence"] / med["batched"], 3), graph_launches=launches,
                invert_batch=Bi, invert_ms=round(inv_ms, 3), invert_ms_min_max=inv_mm, invert_graph_launches=inv_launches,
                morph_rows_kernel=dict(P=Pk, N=N, n=n, L=L, hbm_tb_per_s_datasheet=HBM_TBPS, **kernel),
                morph_rows_slerp_p64_over_batched_morph_p8=round(kernel["slerp"]["ms"] / med["batched"], 6))
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
