"""Time convolution reverb on the GPU: ds_fftconvolve alone at sizes larger than L2 -- a stereo 10-minute piece (9.6 M samples per
channel) with a 3 s stereo IR (48 000 samples, 47 partitions), and a batch of 256 distinct 10 s clips, each with its own 2 s IR --
and render_arrangement(stereo=True) of arrangement_time.py's seeded 4-instrument arrangement with a 3 s stereo IR and sends
(0.2, 0.5, 0.8, 0) against the same call without reverb.

Prints one JSON line (and writes it to --out): the card, its power limit and maximum SM clock read in the same run; device-timed
medians and spreads (CUDA events around each call, which ends in a device synchronise) of the two drop-in workloads alternated in
one process; per-kernel times and launch counts from torch.profiler in a separate run; the bytes the kernels need and the FP32
FMAs of the spectral accumulation over their kernel times, against the B200's 7.7 TB/s HBM3e data-sheet bandwidth and the FP32
FMA bound (148 SMs x 128 FMA per clock x the maximum SM clock); host scipy.signal.fftconvolve (float64) on one item of each
workload; and device-timed medians of --repeats alternated render calls with and without reverb.  Exits non-zero without a CUDA
device.

    python tools_dev/reverb_time.py --out profiles/r10_reverb_time.json"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools_dev"))

from arrangement_time import HBM_TBPS, card  # noqa: E402
from stereo_time import timed  # noqa: E402

SENDS = (0.2, 0.5, 0.8, 0.0)
PANS = (-0.6, -0.2, 0.2, 0.6)
P, NBIN = 1024, 1025
KERNELS = ("conv_forward_kernel", "conv_accumulate_kernel", "conv_output_kernel", "pitch_peak_scale_kernel")


def work(xl, hl, hi):
    """Bytes each kernel needs at the least (every sample, spectrum row and segment read or written once; fp32 samples, complex64
    spectra of 1025 bins per 1024-sample block, fp32 segments of 2048 per 1024 output samples) and the accumulation's FP32 FMAs
    (4 per complex multiply-accumulate, sum over segments of the partitions that meet it, 1025 bins each), for full convolutions."""
    nbx = [-(-n // P) for n in xl]
    Q = [-(-hl[i] // P) for i in hi]
    rows = sum(nbx) + sum(-(-m // P) for m in hl)
    segs = [a + b - 1 for a, b in zip(nbx, Q)]
    cmacs = sum(sum(min(q - 1, s) - max(0, s - (a - 1)) + 1 for s in range(a + q - 1)) for a, q in zip(nbx, Q)) * NBIN
    out = sum(n + hl[i] - 1 for n, i in zip(xl, hi))
    return dict(forward=4.0 * (sum(xl) + sum(hl)) + 8.0 * NBIN * rows,
                accumulate=8.0 * NBIN * rows + 4.0 * 2048 * sum(segs),
                output=4.0 * 2048 * sum(segs) + 4.0 * out), 4.0 * cmacs, out


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--conv-repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("reverb_time: needs a CUDA device", file=sys.stderr)
        return 2
    from scipy.signal import fftconvolve as scipy_fftconvolve
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases

    name, power, clk = card()
    rng = np.random.default_rng(2026)

    def ir(ch, M, seed):
        r = np.random.default_rng(seed)
        return (0.3 * r.standard_normal((ch, M)) * np.exp(-np.arange(M) / (M / 6))).astype(np.float32)

    # ---- the drop-in alone: both workloads larger than L2 ----
    N1, M1 = 16000 * 600, 48000
    stereo_x = torch.randn(2 * N1, device="cuda")
    stereo_h = torch.from_numpy(ir(2, M1, 1)).cuda().reshape(-1)
    B2, N2, M2 = 256, 160000, 32000
    clips_x = torch.randn(B2 * N2, device="cuda")
    clips_h = torch.from_numpy(ir(B2, M2, 2)).cuda().reshape(-1)
    cfg = {"stereo_10min": ([N1, N1], [M1, M1], [0, 1], stereo_x, stereo_h),
           "clips_256x10s": ([N2] * B2, [M2] * B2, list(range(B2)), clips_x, clips_h)}
    outs = {k: torch.empty(sum(n + hl[i] - 1 for n, i in zip(xl, hi)), device="cuda") for k, (xl, hl, hi, _, _) in cfg.items()}

    def call(k, peak=None):
        xl, hl, hi, x, h = cfg[k]
        return codec.fftconvolve_packed(x, xl, h, hl, hi, out=outs[k], target_peak=peak)

    fns = {k: (lambda k=k: call(k)) for k in cfg}
    fns.update({k + "_peak": (lambda k=k: call(k, 0.9)) for k in cfg})
    ms = timed(fns, a.conv_repeats)
    kern = {}
    try:                                                                        # a separate, profiled run per workload
        from torch.profiler import ProfilerActivity, profile
        for k in cfg:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    call(k, 0.9)
                torch.cuda.synchronize()
            d = {}
            for e in prof.events():
                if e.device_type.name != "CUDA":
                    continue
                key = next((kn for kn in KERNELS if kn in e.name), "memcpy" if "emcpy" in e.name else None)
                if key:
                    t = (e.device_time if hasattr(e, "device_time") else e.cuda_time) / 1e3
                    ms_, n_ = d.get(key, (0.0, 0))
                    d[key] = (ms_ + t, n_ + 1)
            kern[k] = {kn: dict(ms_per_call=round(v[0] / 5, 4), launches_per_call=v[1] / 5) for kn, v in d.items()}
    except Exception as ex:
        print(f"reverb_time: profiler run failed: {ex}", file=sys.stderr)
    fma_peak = 148 * 128 * float(clk.split()[0]) * 1e6 if clk and clk.split()[0].replace(".", "").isdigit() else None
    conv = {}
    for k, (xl, hl, hi, x, h) in cfg.items():
        nbytes, fmas, n_out = work(xl, hl, hi)
        entry = dict(items=len(xl), samples_per_item=xl[0], ir_samples=hl[0], outputs=n_out,
                     call_ms=round(float(np.median(ms[k])), 4), call_ms_min_max=[round(min(ms[k]), 4), round(max(ms[k]), 4)],
                     call_ms_peak=round(float(np.median(ms[k + "_peak"])), 4),
                     call_ms_peak_min_max=[round(min(ms[k + "_peak"]), 4), round(max(ms[k + "_peak"]), 4)],
                     kernels=kern.get(k, "not measured"), bytes_needed=nbytes, accumulate_fp32_fma=fmas)
        for kn, short in (("conv_forward_kernel", "forward"), ("conv_accumulate_kernel", "accumulate"), ("conv_output_kernel", "output")):
            t = kern.get(k, {}).get(kn, {}).get("ms_per_call")
            if t:
                bw = nbytes[short] / (t * 1e-3) / 1e12
                entry[short + "_tbps"] = round(bw, 3)
                entry[short + "_share_of_hbm"] = round(bw / HBM_TBPS, 3)
                if short == "accumulate" and fma_peak:
                    entry["accumulate_share_of_fp32_fma_bound"] = round(fmas / (t * 1e-3) / fma_peak, 3)
        xh = x[: xl[0]].cpu().numpy().astype(np.float64)
        hh = h[: hl[0]].cpu().numpy().astype(np.float64)
        t0 = time.perf_counter()
        scipy_fftconvolve(xh, hh)
        entry["scipy_float64_one_item_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        conv[k] = entry

    # ---- the 4-instrument render (arrangement_time.py's draws), stereo, with and without reverb ----
    pool = [0.5, 0.75, 1.0, 1.5, 2.0, 3.0]
    conds, _ = W.synthetic_conditions(4, 512, seed=500)
    tracks = []
    for k in range(4):
        durs = list(rng.choice(pool[:5], 4, replace=False)) + ([3.0] if k % 2 else [])
        notes = [(float(o), float(rng.choice(durs)), int(s), float(g)) for o, s, g in
                 zip(np.sort(rng.uniform(0, 12, 24)), rng.integers(-12, 13, 24), rng.uniform(0.3, 1.0, 24))]
        tracks.append((cases.vq_latents(B=1, seed=40 + k).cuda(), conds[k:k + 1].cuda(), notes, float(rng.uniform(0.5, 1.0)), 0.05,
                       PANS[k]))
    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    room = torch.from_numpy(ir(2, M1, 3)).cuda()
    rms = timed({"reverb": lambda: pipe.render_arrangement(tracks, sample_steps=a.steps, target_peak=0.9, stereo=True,
                                                           impulse_response=room, reverb_sends=list(SENDS)),
                 "dry": lambda: pipe.render_arrangement(tracks, sample_steps=a.steps, target_peak=0.9, stereo=True)}, a.repeats)
    plan = TextToTimbre.arrangement_plan(tracks)
    line = dict(tool="reverb_time", card=name, power_limit=power, max_sm_clock=clk, convolve=conv,
                convolve_note="host plan + one metadata copy + kernels, CUDA events around the call, the workloads alternated",
                render=dict(tracks=len(tracks), pans=list(PANS), sends=list(SENDS), ir_samples=M1, notes=len(plan.note_item),
                            track_samples=int(plan.track_len), sample_steps=a.steps, repeats=a.repeats,
                            weights="deployed architecture, random init, default tiling policy",
                            ms={k: round(float(np.median(v)), 2) for k, v in rms.items()},
                            ms_min_max={k: [round(min(v), 2), round(max(v), 2)] for k, v in rms.items()}),
                hbm_datasheet_tbps=HBM_TBPS, fp32_fma_bound_per_s=fma_peak)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
