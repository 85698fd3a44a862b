"""Time the upload resampler (ds_resample) on the GPU: 1024 distinct 4.08 s clips, half at 44.1 kHz and half at 48 kHz (about 770 MB
of fp32 input, more than the L2 holds), peak-normalised and resampled to 16 kHz with a fixed length of 65 280 samples, as
TextToTimbre.encode_audio does for a batch of uploads.  Prints one JSON line (and writes it to --out): the card, its power limit and
maximum SM clock read in the same run; the device-timed median of --repeats calls (CUDA events, after a warm-up) through the
polyphase-table path and through the direct path (DS_RESAMPLE_DIRECT=1) on the same batch, and whether the two agree bit for bit;
per-kernel times from torch.profiler in a separate run; taps and bytes per kernel with the achieved rates and the bounds they are
measured against; and, as host reference points, scipy.signal.resample_poly and the float64 oracle per clip.  Exits non-zero
without a CUDA device.

    python tools_dev/resample_time.py --out profiles/resample_time.json"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OUT_LEN = 65280
RATES = (44100, 48000)


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
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("resample_time: needs a CUDA device", file=sys.stderr)
        return 2
    from diffusynth_b200 import codec
    from tests import resample_oracle as P

    srs = [RATES[k * len(RATES) // a.clips] for k in range(a.clips)]
    lengths = [int(np.ceil(OUT_LEN * sr / 16000)) for sr in srs]              # 4.08 s at each rate
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    packed = 0.3 * torch.randn((sum(lengths),), device="cuda", generator=g)    # distinct clips, generated on the device
    out = torch.empty((a.clips * OUT_LEN,), dtype=torch.float32, device="cuda")

    def run():
        codec.resample_packed(packed, lengths, srs, 16000, out_lengths=OUT_LEN, normalize_peak=True, out=out)

    def timed():
        run()                                                                   # warm-up
        torch.cuda.synchronize()
        ms = []
        for _ in range(a.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), [round(min(ms), 3), round(max(ms), 3)]

    table_ms, table_mm = timed()
    table_out = out.clone()
    os.environ["DS_RESAMPLE_DIRECT"] = "1"
    direct_ms, direct_mm = timed()
    del os.environ["DS_RESAMPLE_DIRECT"]
    identical = bool(torch.equal(out, table_out))

    kernels = {}
    try:                                                                        # a separate, profiled run of the table path
        from torch.profiler import ProfilerActivity, profile
        run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run()
            torch.cuda.synchronize()
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            key = next((k for k in ("resample_table_kernel", "resample_peak_kernel", "resample_kernel") if k in e.name),
                       "memcpy" if "emcpy" in e.name else None)
            if key:
                kernels[key] = kernels.get(key, 0.0) + getattr(e, "device_time", getattr(e, "cuda_time", 0.0)) / 1e3   # us -> ms
    except Exception as ex:
        print(f"resample_time: profiler run failed: {ex}", file=sys.stderr)

    # work per kernel, from the shapes: the table path sums taps4 = 2F+2 rounded up to 4 products per output (2F+2 of them inside
    # the filter's support or its zero-padded edge)
    def taps(sr, rounded):
        F = int(np.floor(64 / (16000 / sr)))
        return ((2 * F + 2 + 3) // 4 * 4) if rounded else 2 * F + 2
    n_valid = [P.resample_length(n, sr, 16000) for n, sr in zip(lengths, srs)]
    fma_exec = sum(min(v, OUT_LEN) * taps(sr, True) for v, sr in zip(n_valid, srs))
    fma_filter = sum(min(v, OUT_LEN) * taps(sr, False) for v, sr in zip(n_valid, srs))
    in_bytes, out_bytes = 4 * sum(lengths), 4 * a.clips * OUT_LEN
    name, power, clk = card()
    try:
        clk_hz = float(clk.split()[0]) * 1e6
    except Exception:
        clk_hz = None
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rk = kernels.get("resample_kernel")
    rates = {}
    if rk:
        rates["resample_kernel_taps_per_s"] = fma_exec / (rk * 1e-3)
        if clk_hz:
            rates["fp32_fma_bound_per_s"] = sms * 128 * clk_hz                  # 128 FP32 FMA per SM per clock at the max SM clock
            rates["lds_bound_taps_per_s"] = sms * 32 * clk_hz                   # one 4-byte shared-memory load per tap: 128 B per SM per clock
            rates["share_of_lds_bound"] = rates["resample_kernel_taps_per_s"] / rates["lds_bound_taps_per_s"]
            rates["share_of_fma_bound"] = rates["resample_kernel_taps_per_s"] / rates["fp32_fma_bound_per_s"]
        rates["resample_kernel_bytes_per_s"] = (in_bytes + out_bytes) / (rk * 1e-3)
    pk = kernels.get("resample_peak_kernel")
    if pk:
        rates["peak_kernel_bytes_per_s"] = in_bytes / (pk * 1e-3)
    rates["hbm_bound_bytes_per_s"] = 7.7e12                                     # HGX B200 data sheet, per GPU

    # host reference points: one clip per rate
    from scipy.signal import resample_poly
    rng = np.random.default_rng(0)
    host = {}
    for sr in RATES:
        x = rng.standard_normal(int(np.ceil(OUT_LEN * sr / 16000))).astype(np.float32)
        up, down = 16000 // np.gcd(sr, 16000), sr // np.gcd(sr, 16000)
        t0 = time.perf_counter()
        for _ in range(10):
            resample_poly(x / np.abs(x).max(), up, down)
        host[f"resample_poly_ms_per_clip_{sr}"] = round((time.perf_counter() - t0) / 10 * 1e3, 3)
        t0 = time.perf_counter()
        P.resample(x.astype(np.float64) / np.abs(x).max(), sr, 16000)
        host[f"oracle_f64_ms_per_clip_{sr}"] = round((time.perf_counter() - t0) * 1e3, 1)

    line = dict(tool="resample_time", card=name, power_limit=power, max_sm_clock=clk, clips=a.clips, rates_in=list(RATES),
                input_samples=sum(lengths), input_mb=round(in_bytes / 1e6, 1), out_len=OUT_LEN, normalize_peak=True,
                repeats=a.repeats, l2_note="input larger than the 126 MB L2; the same buffers are reused between runs",
                table_path_ms=round(table_ms, 3), table_path_ms_min_max=table_mm,
                direct_path_ms=round(direct_ms, 3), direct_path_ms_min_max=direct_mm, direct_equals_table_bitwise=identical,
                kernel_ms_profiled={k: round(v, 4) for k, v in kernels.items()} or "not measured",
                taps_executed=fma_exec, taps_in_filter=fma_filter, input_bytes=in_bytes, output_bytes=out_bytes,
                achieved=rates, host_reference=host, host_reference_note="one CPU thread per clip, this run's host")
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
