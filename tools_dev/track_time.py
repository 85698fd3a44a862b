"""Time one note arrangement end to end on the GPU (TextToTimbre.render_track's two stages) and the float64 CPU oracle of its
pitch-shift + mix stage.  A fixed, seeded track with the deployed architecture at random init: 64 notes, 8 distinct durations from
0.5 s to 3 s, semitones in [-12, 12], overlapping onsets.  Prints one JSON line (and writes it to --out): the card and its power
limit read in the same run, the distinct-duration / distinct-pair counts, device-timed synthesis and pitch + mix (CUDA events,
median of --repeats after a warm-up), the kernels and copies of the pitch/mix stage (torch.profiler, separate run), the host-timed
oracle pitch + mix, and the track's rel-L2 against that oracle.  Exits non-zero without a CUDA device.

    python tools_dev/track_time.py --out profiles/track_time.json"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1] if len(q) > 1 else "not measured"
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "not measured"


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("track_time: needs a CUDA device", file=sys.stderr)
        return 2
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases
    from tests import pitch_oracle as P

    rng = np.random.default_rng(2024)
    durs = np.round(np.linspace(0.5, 3.0, 8), 4)
    notes = [(float(on), float(durs[i % 8]), int(s), float(g)) for i, (on, s, g) in
             enumerate(zip(np.sort(rng.uniform(0, 24, 64)), rng.integers(-12, 13, 64), rng.uniform(0.3, 1.0, 64)))]
    plan = TextToTimbre.track_plan(notes)
    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    cond, _ = W.synthetic_conditions(1, 512)
    inst, cond = cases.vq_latents(B=1, seed=22).cuda(), cond.cuda()

    def synth():
        return pipe.synthesize_notes(inst, cond, plan.durations, sample_steps=a.steps)

    timbres = synth()                                                           # warm-up: builds one graph per distinct width
    sources = [timbres[d].waveforms[0] for d, _ in plan.pairs]
    semis = [s for _, s in plan.pairs]

    def shift_mix():
        return codec.shift_and_mix(sources, semis, plan.note_pair, plan.onsets, plan.gains)

    track = shift_mix()
    torch.cuda.synchronize()

    def timed(fn):
        ms = []
        for _ in range(a.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), ms

    synth_ms, _ = timed(synth)
    pm_ms, pm_all = timed(shift_mix)

    kernels = copies = None
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            shift_mix()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
        kernels = sum(1 for n in names if "pitch_" in n)
        copies = sum(1 for n in names if "Memcpy" in n or "memcpy" in n)
    except Exception as e:                                                      # the count is then reported as not measured
        print(f"track_time: profiler count failed: {e}", file=sys.stderr)

    waves = [t.waveforms[0].cpu().numpy().astype(np.float64) for t in timbres]
    t0 = time.perf_counter()
    shifted = [P.pitch_shift(waves[d], s) for d, s in plan.pairs]
    ref = P.mix_track([shifted[p] for p in plan.note_pair], plan.onsets, plan.gains)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    got = track.cpu().numpy().astype(np.float64)
    name, power = card()
    line = dict(tool="track_time", card=name, power_limit=power, notes=len(notes), distinct_durations=len(plan.durations),
                distinct_widths=len({TextToTimbre.note_width(d) for d in plan.durations}), distinct_pairs=len(plan.pairs),
                track_samples=int(track.numel()), sample_steps=a.steps, repeats=a.repeats,
                synthesis_ms=round(synth_ms, 3), pitch_mix_ms=round(pm_ms, 3),
                pitch_mix_ms_min_max=[round(min(pm_all), 3), round(max(pm_all), 3)],
                pitch_mix_kernels=kernels if kernels is not None else "not measured",
                pitch_mix_copies=copies if copies is not None else "not measured",
                pitch_mix_library_calls=4, cpu_oracle_pitch_mix_ms=round(cpu_ms, 1), cpu_oracle_runs=1,
                track_rel_l2_vs_oracle=float(np.linalg.norm(got - ref) / np.linalg.norm(ref)))
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
