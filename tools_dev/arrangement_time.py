"""Time a multi-instrument arrangement on the GPU: TextToTimbre.render_arrangement against the per-track loop a caller would
otherwise write (render_track per instrument, then a torch sum of the tracks), and the arrangement mix (ds_mix_arrangement) alone on
a mix of several thousand distinct notes, large enough to leave L2.

The arrangement is seeded and is what a user would write: 4 instruments (own latent and condition each) x 24 notes over 12 s,
each track using 4 or 5 durations out of a shared pool of 6, semitones in [-12, 12], a 50 ms fade and a peak of 0.9 for the
timed arrangement (the loop has neither, as render_track offers neither).  Deployed architecture at
random init, 20 DDIM steps, the default tiling policy.  Prints one JSON line (and writes it to --out): the card, its power limit and
maximum SM clock read in the same run; the device-timed medians (CUDA events around each call, which ends in a device synchronise)
of --repeats calls of each, alternating the two; the graph launches of each; the rel-L2 between the loop's sum and a fade-free,
unnormalised render_arrangement; and, for the mix alone, the
call's device-timed median (with fades, with fades and a peak, and as mix_track: the same notes without fades), its kernels' times from torch.profiler in a separate run, and the bytes the mix needs (every note sample
read once, the track written once; the normalisation reads and writes the track again) over the kernel time, against the
B200's 7.7 TB/s HBM3e data-sheet bandwidth.  Exits non-zero without a CUDA device.

    python tools_dev/arrangement_time.py --out profiles/arrangement_time.json"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1] if len(q) > 1 else "not measured", q[2] if len(q) > 2 else "not measured"
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "not measured", "not measured"


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--mix-notes", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("arrangement_time: needs a CUDA device", file=sys.stderr)
        return 2
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases

    rng = np.random.default_rng(2026)
    pool = [0.5, 0.75, 1.0, 1.5, 2.0, 3.0]
    conds, _ = W.synthetic_conditions(4, 512, seed=500)
    tracks = []
    for k in range(4):
        durs = list(rng.choice(pool[:5], 4, replace=False)) + ([3.0] if k % 2 else [])
        notes = [(float(o), float(rng.choice(durs)), int(s), float(g)) for o, s, g in
                 zip(np.sort(rng.uniform(0, 12, 24)), rng.integers(-12, 13, 24), rng.uniform(0.3, 1.0, 24))]
        tracks.append((cases.vq_latents(B=1, seed=40 + k).cuda(), conds[k:k + 1].cuda(), notes, float(rng.uniform(0.5, 1.0)), 0.05))
    plan = TextToTimbre.arrangement_plan(tracks)
    per_track_widths = [len({TextToTimbre.note_width(d) for _, d, _, _ in t[2]}) for t in tracks]

    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    groups = [0]
    inner = pipe._run

    def counted(*args, **kw):                                                   # one _run = one graph launch
        groups[0] += 1
        return inner(*args, **kw)
    pipe._run = counted

    def arrangement():
        return pipe.render_arrangement(tracks, sample_steps=a.steps, target_peak=0.9)

    def loop(feeds=(None,) * len(tracks)):
        outs = [pipe.render_track(lat, cond, [(o, d, s, g * gain) for o, d, s, g in notes], sample_steps=a.steps, noise_feeds=f)
                for (lat, cond, notes, gain, _), f in zip(tracks, feeds)]
        total = torch.zeros(max(x.numel() for x in outs), device="cuda")
        for x in outs:
            total[:x.numel()] += x
        return total

    runs = {"render_arrangement": arrangement, "render_track_loop": loop}
    outs, launches = {}, {}
    for name, fn in runs.items():                                               # warm-up: samplers, graphs, buffers
        groups[0] = 0
        outs[name] = fn()
        launches[name] = groups[0]
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    for _ in range(a.repeats):
        for k, fn in runs.items():                                              # alternate the two
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    # same work and the same noise (one feed per row) as the loop, no fade, no peak, untimed: the rows run at other batch sizes, so
    # the default tiling policy rounds them differently (batch_invariant=True makes them agree to the summation order,
    # tests/test_gpu_arrangement.py)
    feeds = [W.host_noise(900 + r, 1 + a.steps, 1) for r in range(len(plan.rows))]
    plain = pipe.render_arrangement([(lat, cond, notes, gain, 0.0) for lat, cond, notes, gain, _ in tracks], sample_steps=a.steps,
                                    noise_feeds=feeds)
    x = plain.double()
    y = loop([[feeds[r] for r, (k, _) in enumerate(plan.rows) if k == t] for t in range(len(tracks))]).double()
    arr_vs_loop = float((x - y).norm() / y.norm())

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

    def mix(peak):
        return codec.mix_arrangement(src, offs, lengths, onsets, gains, fades, target_peak=peak, track_len=track_len)

    mix_ms = {}
    for name, fn in (("plain", lambda: mix(None)), ("peak", lambda: mix(0.9)),
                     ("track", lambda: codec.mix_track(src, offs, lengths, onsets, gains, track_len=track_len))):
        fn()
        torch.cuda.synchronize()
        t = []
        for _ in range(20):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            t.append(e0.elapsed_time(e1))
        mix_ms[name] = t
    kern = {}
    try:                                                                        # a separate, profiled run
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                mix(0.9)
            torch.cuda.synchronize()
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            key = next((k for k in ("pitch_arrange_kernel", "pitch_peak_scale_kernel") if k in e.name), "memcpy" if "emcpy" in e.name else None)
            if key:
                kern[key] = kern.get(key, 0.0) + (e.device_time if hasattr(e, "device_time") else e.cuda_time) / 1e3 / 5   # us -> ms per call
    except Exception as ex:
        print(f"arrangement_time: profiler run failed: {ex}", file=sys.stderr)
    mix_bytes = 4.0 * (K * L + track_len)
    scale_bytes = 8.0 * track_len
    mix_line = dict(notes=K, note_samples=L, track_samples=track_len, source_mb=round(K * L * 4 / 1e6, 1),
                    call_ms_plain=round(float(np.median(mix_ms["plain"])), 4), call_ms_peak=round(float(np.median(mix_ms["peak"])), 4),
                    call_ms_track=round(float(np.median(mix_ms["track"])), 4),
                    call_note="host plan + one metadata copy + kernels, CUDA events around the call",
                    kernel_ms_profiled={k: round(v, 4) for k, v in kern.items()} or "not measured")
    if "pitch_arrange_kernel" in kern:
        bw = mix_bytes / (kern["pitch_arrange_kernel"] * 1e-3) / 1e12
        mix_line.update(arrange_kernel_bytes=mix_bytes, arrange_kernel_tbps=round(bw, 3), arrange_kernel_share_of_hbm=round(bw / HBM_TBPS, 3))
    if "pitch_peak_scale_kernel" in kern:
        bw = scale_bytes / (kern["pitch_peak_scale_kernel"] * 1e-3) / 1e12
        mix_line.update(peak_scale_kernel_bytes=scale_bytes, peak_scale_kernel_tbps=round(bw, 3))

    name, power, clk = card()
    line = dict(tool="arrangement_time", card=name, power_limit=power, max_sm_clock=clk, tracks=len(tracks),
                notes=len(plan.note_item), rows=len(plan.rows), distinct_widths=len(set(plan.widths)),
                per_track_distinct_widths=per_track_widths, pitch_items=len(plan.items), track_samples=int(plan.track_len),
                sample_steps=a.steps, repeats=a.repeats, weights="deployed architecture, random init, default tiling policy",
                graph_launches=launches,
                render_arrangement_ms=round(med["render_arrangement"], 2),
                render_arrangement_ms_min_max=[round(min(ms["render_arrangement"]), 2), round(max(ms["render_arrangement"]), 2)],
                render_track_loop_ms=round(med["render_track_loop"], 2),
                render_track_loop_ms_min_max=[round(min(ms["render_track_loop"]), 2), round(max(ms["render_track_loop"]), 2)],
                speedup=round(med["render_track_loop"] / med["render_arrangement"], 3),
                arrangement_vs_loop_rel_l2=arr_vs_loop,
                arrangement_vs_loop_note="render_arrangement without fades or peak against the loop's sum, same noise feeds; default tiling policy",
                mix=mix_line, hbm_datasheet_tbps=HBM_TBPS)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
