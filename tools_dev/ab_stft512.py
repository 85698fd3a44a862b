"""A/B check of the n_fft-1024 STFT kernels between two builds: runs ds_stft_decode_istft and ds_stft_encode of this tree's library
and of another build (e.g. the parent commit's, --other-lib PATH) on one seeded input in the same process pair and compares the
outputs bit for bit.  Prints one JSON line; exits non-zero on a difference or without a CUDA device.

    python tools_dev/ab_stft512.py --other-lib /path/to/parent/libdiffusynth_b200.so"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run_one(out_path: str) -> None:
    import numpy as np
    import torch
    from diffusynth_b200 import codec
    assert torch.cuda.is_available(), "needs a CUDA device"
    g = torch.Generator().manual_seed(1234)
    B, T = 3, 256
    spec = torch.stack([torch.rand((B, 512, T), generator=g) * 3, torch.randn((B, 512, T), generator=g),
                        torch.randn((B, 512, T), generator=g)], dim=1).cuda()
    wave = codec.spectrogram_to_waveform(spec)                               # ds_stft_decode_istft
    enc = codec.waveform_to_spectrogram(wave, time_resolution=T)             # ds_stft_encode
    torch.cuda.synchronize()
    np.savez(out_path, wave=wave.cpu().numpy(), enc=enc.cpu().numpy())


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--other-lib", required=True)
    ap.add_argument("--child", default=None)
    a = ap.parse_args()
    if a.child:
        run_one(a.child)
        return 0
    import numpy as np
    from diffusynth_b200 import _build
    _build.build()
    res = {}
    with tempfile.TemporaryDirectory() as d:
        for name, lib in (("this", _build.LIB), ("other", os.path.abspath(a.other_lib))):
            env = dict(os.environ, DS_LIB_PATH=lib)
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--other-lib", a.other_lib, "--child", os.path.join(d, name + ".npz")],
                                  env=env)
            res[name] = dict(np.load(os.path.join(d, name + ".npz")))
    same = {k: bool(np.array_equal(res["this"][k].view(np.uint32), res["other"][k].view(np.uint32))) for k in ("wave", "enc")}
    print(json.dumps(dict(check="stft512_bit_identity", ds_stft_decode_istft=same["wave"], ds_stft_encode=same["enc"],
                          samples=int(res["this"]["wave"].size), spec_values=int(res["this"]["enc"].size))))
    return 0 if all(same.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
