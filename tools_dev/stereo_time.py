"""Time stereo arrangements on the GPU against mono: the stereo mix (ds_mix_stereo) against the arrangement mix
(ds_mix_arrangement) on arrangement_time.py's 4096-note, 10-minute set, and render_arrangement(stereo=True) against the mono render
of arrangement_time.py's seeded 4-instrument arrangement, each track panned (-0.6, -0.2, 0.2, 0.6).

Prints one JSON line (and writes it to --out): the card, its power limit and maximum SM clock read in the same run; for the mix
alone, device-timed medians (CUDA events around each call, which ends in a device synchronise) of mono and stereo calls alternated
in one process, with fades, with and without a peak of 0.9; the kernels' times from torch.profiler in a separate run; and the bytes
each arrange kernel needs (every note sample read once, every output channel written once) over its kernel time, against the
B200's 7.7 TB/s HBM3e data-sheet bandwidth.  For the render, device-timed medians of --repeats alternated stereo and mono calls,
with a 50 ms fade and a peak of 0.9 (deployed architecture at random init, 20 DDIM steps, the default tiling policy).  Exits
non-zero without a CUDA device.

    python tools_dev/stereo_time.py --out profiles/r09_stereo_time.json"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools_dev"))

from arrangement_time import HBM_TBPS, card  # noqa: E402

PANS = (-0.6, -0.2, 0.2, 0.6)


def timed(fns: dict, repeats: int) -> dict:
    """Device-timed milliseconds of each call, the calls alternated; one untimed warm-up call of each first."""
    import torch
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(repeats):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    return ms


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--mix-repeats", type=int, default=20)
    ap.add_argument("--mix-notes", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("stereo_time: needs a CUDA device", file=sys.stderr)
        return 2
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases

    # ---- the arrangement of arrangement_time.py (same seed, same draws), each track panned ----
    rng = np.random.default_rng(2026)
    pool = [0.5, 0.75, 1.0, 1.5, 2.0, 3.0]
    conds, _ = W.synthetic_conditions(4, 512, seed=500)
    tracks = []
    for k in range(4):
        durs = list(rng.choice(pool[:5], 4, replace=False)) + ([3.0] if k % 2 else [])
        notes = [(float(o), float(rng.choice(durs)), int(s), float(g)) for o, s, g in
                 zip(np.sort(rng.uniform(0, 12, 24)), rng.integers(-12, 13, 24), rng.uniform(0.3, 1.0, 24))]
        tracks.append((cases.vq_latents(B=1, seed=40 + k).cuda(), conds[k:k + 1].cuda(), notes, float(rng.uniform(0.5, 1.0)), 0.05,
                       PANS[k]))

    # ---- the mix alone: distinct sources per note (not L2-resident), 10 minutes of track ----
    K = a.mix_notes
    L = 256 * (4 * 48 - 1)
    track_len = 16000 * 600
    src = torch.randn(K * L, device="cuda")
    offs = np.arange(K, dtype=np.int64) * L
    onsets = rng.integers(0, track_len - L, K)
    gains = rng.uniform(-1, 1, K).astype(np.float32)
    fades = np.full(K, 800, dtype=np.int64)
    lengths = np.full(K, L, dtype=np.int64)
    pans = rng.uniform(-1, 1, K).astype(np.float32)

    def mono(peak):
        return codec.mix_arrangement(src, offs, lengths, onsets, gains, fades, target_peak=peak, track_len=track_len)

    def stereo(peak):
        return codec.mix_stereo(src, offs, lengths, onsets, gains, pans, fades, target_peak=peak, track_len=track_len)

    mix_ms = timed({"mono": lambda: mono(None), "stereo": lambda: stereo(None), "mono_peak": lambda: mono(0.9),
                    "stereo_peak": lambda: stereo(0.9)}, a.mix_repeats)
    kern = {}
    try:                                                                        # a separate, profiled run per channel count
        from torch.profiler import ProfilerActivity, profile
        for tag, fn in (("mono", mono), ("stereo", stereo)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    fn(0.9)
                torch.cuda.synchronize()
            for e in prof.events():
                if e.device_type.name != "CUDA":
                    continue
                key = next((k for k in ("pitch_arrange_kernel", "pitch_peak_scale_kernel") if k in e.name),
                           "memcpy" if "emcpy" in e.name else None)
                if key:
                    t = (e.device_time if hasattr(e, "device_time") else e.cuda_time) / 1e3 / 5       # us -> ms per call
                    kern.setdefault(tag, {})[key] = kern.get(tag, {}).get(key, 0.0) + t
    except Exception as ex:
        print(f"stereo_time: profiler run failed: {ex}", file=sys.stderr)
    mix_line = dict(notes=K, note_samples=L, track_samples=track_len, source_mb=round(K * L * 4 / 1e6, 1),
                    call_ms={k: round(float(np.median(v)), 4) for k, v in mix_ms.items()},
                    call_ms_min_max={k: [round(min(v), 4), round(max(v), 4)] for k, v in mix_ms.items()},
                    call_note="host plan + one metadata copy + kernels, CUDA events around the call, mono and stereo alternated",
                    kernel_ms_profiled={t: {k: round(v, 4) for k, v in d.items()} for t, d in kern.items()} or "not measured")
    for tag, ch in (("mono", 1), ("stereo", 2)):
        ms = kern.get(tag, {}).get("pitch_arrange_kernel")
        if ms:
            nbytes = 4.0 * (K * L + ch * track_len)
            bw = nbytes / (ms * 1e-3) / 1e12
            mix_line[f"{tag}_arrange_kernel"] = dict(bytes=nbytes, tbps=round(bw, 3), share_of_hbm=round(bw / HBM_TBPS, 3))
    if all(kern.get(t, {}).get("pitch_arrange_kernel") for t in ("mono", "stereo")):
        mix_line["stereo_over_mono_kernel"] = round(kern["stereo"]["pitch_arrange_kernel"] / kern["mono"]["pitch_arrange_kernel"], 3)

    # ---- the 4-instrument render, stereo against mono ----
    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    ms = timed({"stereo": lambda: pipe.render_arrangement(tracks, sample_steps=a.steps, target_peak=0.9, stereo=True),
                "mono": lambda: pipe.render_arrangement([t[:5] for t in tracks], sample_steps=a.steps, target_peak=0.9)}, a.repeats)
    plan = TextToTimbre.arrangement_plan(tracks)
    name, power, clk = card()
    line = dict(tool="stereo_time", card=name, power_limit=power, max_sm_clock=clk, mix=mix_line,
                render=dict(tracks=len(tracks), pans=list(PANS), notes=len(plan.note_item), track_samples=int(plan.track_len),
                            sample_steps=a.steps, repeats=a.repeats, weights="deployed architecture, random init, default tiling policy",
                            ms={k: round(float(np.median(v)), 2) for k, v in ms.items()},
                            ms_min_max={k: [round(min(v), 2), round(max(v), 2)] for k, v in ms.items()}),
                hbm_datasheet_tbps=HBM_TBPS)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
