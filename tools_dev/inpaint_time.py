"""Time inpainting with text on the GPU: TextToTimbre.inpaint against TextToTimbre.generate at B = 64, w = 64 and 20 DDIM steps with
CFG 6 (deployed architecture, random-init weights), and the mask zoom (ds_mask_zoom) alone for 64 distinct 513 x 257 masks.
inpaint takes its 64 masks as host numpy arrays, as an upload handler holds them, so its time includes their copy to the device
and the zoom.  Prints one JSON line (and writes it to --out): the card, its power limit and maximum SM clock read in the same run;
the device-timed medians (CUDA events around each call, after a warm-up) of --repeats calls of each pipeline, alternating the two;
the zoom's device-timed median and its kernels from torch.profiler in a separate run; and, as the host reference point, one
scipy.ndimage.zoom of a 513 x 257 mask on this run's host.  Exits non-zero without a CUDA device.

    python tools_dev/inpaint_time.py --out profiles/inpaint_time.json"""
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1] if len(q) > 1 else "not measured", q[2] if len(q) > 2 else "not measured"
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "not measured", "not measured"


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("inpaint_time: needs a CUDA device", file=sys.stderr)
        return 2
    import scipy.ndimage as nd
    from diffusynth_b200 import TextToTimbre, codec, weights as W
    from oracle import cases

    B, width = a.batch, 64
    rng = np.random.default_rng(6)
    masks = []
    for _ in range(B):                                                          # keep the upload except one time-frequency region
        m = np.ones((513, 257), np.float32)
        f0, t0 = rng.integers(0, 300), rng.integers(0, 150)
        m[f0: f0 + rng.integers(60, 200), t0: t0 + rng.integers(40, 100)] = 0.0
        masks.append(m)
    pipe = TextToTimbre.random_init(device="cuda", seed=0)
    cond, uncond = W.synthetic_conditions(B, 512)
    cond, uncond = cond.cuda(), uncond.cuda()
    guide = pipe.encode_audio(torch.from_numpy(cases.synthetic_wave(seed=33)).float()[None].cuda(), width=width)

    runs = {"generate": lambda: pipe.generate(cond, uncond, steps=a.steps, cfg_scale=6, width=width, seed=0),
            "inpaint": lambda: pipe.inpaint(guide, masks, cond, uncond, steps=a.steps, cfg_scale=6, seed=0)}
    for fn in runs.values():                                                    # warm-up: samplers, graphs, buffers
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in runs}
    launches = {}
    for _ in range(a.repeats):
        for k, fn in runs.items():                                              # alternate the two
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
            launches[k] = pipe.last_launches
    med = {k: float(np.median(v)) for k, v in ms.items()}

    packed = torch.from_numpy(np.concatenate([m.reshape(-1) for m in masks])).cuda()
    zoomed = torch.empty((B, 1, 128, width), dtype=torch.float32, device="cuda")

    def zoom():
        codec.zoom_packed(packed, [(513, 257)] * B, (128, width), out=zoomed)

    zoom()
    torch.cuda.synchronize()
    zms = []
    for _ in range(max(a.repeats, 20)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        zoom()
        e1.record()
        e1.synchronize()
        zms.append(e0.elapsed_time(e1))
    kernels = {}
    try:                                                                        # a separate, profiled run of the zoom
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            zoom()
            torch.cuda.synchronize()
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            key = next((k for k in ("zoom_cols_kernel", "zoom_rows_kernel") if k in e.name), "memcpy" if "emcpy" in e.name else None)
            if key:
                kernels[key] = kernels.get(key, 0.0) + getattr(e, "device_time", getattr(e, "cuda_time", 0.0)) / 1e3   # us -> ms
    except Exception as ex:
        print(f"inpaint_time: profiler run failed: {ex}", file=sys.stderr)
    ref = np.stack([nd.zoom(m, (128 / 513, width / 257)) for m in masks[:4]])
    zoom_err = float(np.abs(zoomed[:4, 0].cpu().numpy().astype(np.float64) - ref).max())

    t0 = time.perf_counter()
    for m in masks[:20]:
        nd.zoom(m, (128 / 513, width / 257))
    host_ms = (time.perf_counter() - t0) / 20 * 1e3

    name, power, clk = card()
    line = dict(tool="inpaint_time", card=name, power_limit=power, max_sm_clock=clk, batch=B, width=width, steps=a.steps, cfg_scale=6,
                sampler="ddim", repeats=a.repeats, weights="deployed architecture, random init",
                generate_ms=round(med["generate"], 3), generate_ms_min_max=[round(min(ms["generate"]), 3), round(max(ms["generate"]), 3)],
                inpaint_ms=round(med["inpaint"], 3), inpaint_ms_min_max=[round(min(ms["inpaint"]), 3), round(max(ms["inpaint"]), 3)],
                inpaint_over_generate=round(med["inpaint"] / med["generate"], 4), graph_launches=launches,
                inpaint_note="masks passed as host numpy arrays: the time includes their copy to the device and the zoom",
                mask_zoom_masks=B, mask_zoom_shape="513x257 -> 128x64", mask_zoom_ms=round(float(np.median(zms)), 4),
                mask_zoom_ms_min_max=[round(min(zms), 4), round(max(zms), 4)],
                mask_zoom_kernel_ms_profiled={k: round(v, 4) for k, v in kernels.items()} or "not measured",
                mask_zoom_max_abs_err_vs_scipy=zoom_err,
                host_scipy_zoom_ms_per_mask=round(host_ms, 3), host_reference_note="scipy.ndimage.zoom, one CPU thread, this run's host")
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
