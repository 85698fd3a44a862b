"""Sample-rate conversion on the GPU (ds_resample): a ragged batch of clips at common rates against the float64 oracle
(tests/resample_oracle.py), the direct path of pairs above the table cap, normalisation / crop / zero-pad, determinism, the
codec.resample drop-in, and TextToTimbre.encode_audio / modify with uploads at any sample rate."""
import os

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec, weights as W
from diffusynth_b200.codec import adjust_audio_length, waveform_to_spectrogram
from tests import resample_oracle as P
from tests.gpu_util import rel

pytestmark = pytest.mark.gpu

RATES_IN = [8000, 11025, 16000, 22050, 32000, 44100, 48000, 96000]
PAIRS = [(o, 16000) for o in RATES_IN] + [(16000, 44100), (16000, 48000)]


def _clip(sr, n, seed):
    """A few partials below 0.45 * min(sr, 16 kHz) with a decay, plus a little noise; n samples at sr."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    f_top = 0.45 * min(sr, 16000)
    y = sum(a * np.sin(2 * np.pi * f * t + p) for a, f, p in zip(rng.uniform(0.2, 1, 4), rng.uniform(50, f_top, 4), rng.uniform(0, 6, 4)))
    return (2.5 * y * np.exp(-2 * t) + 0.02 * rng.standard_normal(n)).astype(np.float32)


def _batch():
    """Ragged: clip k lasts 0.25 .. 0.6 s at its input rate."""
    clips = [_clip(o, int(o * (0.25 + 0.05 * k)) + 17 * k, 40 + k) for k, (o, _) in enumerate(PAIRS)]
    return clips, [o for o, _ in PAIRS], [t for _, t in PAIRS]


def _packed(clips):
    return torch.from_numpy(np.concatenate(clips)).cuda(), [len(c) for c in clips]


def _split(out, lens):
    return [p.cpu().numpy().astype(np.float64) for p in torch.split(out, lens)]


def crel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def test_ragged_batch_against_oracle():
    clips, o, t = _batch()
    packed, lengths = _packed(clips)
    out = codec.resample_packed(packed, lengths, o, t)
    n_out = [P.resample_length(n, a, b) for n, a, b in zip(lengths, o, t)]
    assert out.numel() == sum(n_out)
    worst = 0.0
    for y, a, b, got in zip(clips, o, t, _split(out, n_out)):
        e = crel(got, P.resample(y.astype(np.float64), a, b))
        print(f"\n{a} -> {b}: {len(y)} -> {len(got)} samples, rel-L2 vs oracle {e:.2e}")
        worst = max(worst, e)
        if a == b:
            assert np.array_equal(got, y.astype(np.float64))
    assert worst <= 1e-5, worst


def test_direct_path_above_the_table_cap_and_bit_identical_to_the_table_path():
    """44101 -> 16000 has up = 16000 phases: its table (16000 x 356 coefficients) is above the cap, so it is evaluated per tap.
    Forcing every pair onto the direct path (DS_RESAMPLE_DIRECT=1) reproduces the table path bit for bit."""
    y = _clip(44101, 20000, 7)
    got = codec.resample_packed(torch.from_numpy(y).cuda(), [len(y)], 44101, 16000).cpu().numpy().astype(np.float64)
    e = crel(got, P.resample(y.astype(np.float64), 44101, 16000))
    print(f"\n44101 -> 16000 (direct path): rel-L2 vs oracle {e:.2e}")
    assert len(got) == P.resample_length(len(y), 44101, 16000) and e <= 1e-5
    clips, o, t = _batch()
    packed, lengths = _packed(clips)
    table = codec.resample_packed(packed, lengths, o, t, out_lengths=[3000] * len(clips), normalize_peak=True)
    os.environ["DS_RESAMPLE_DIRECT"] = "1"
    try:
        direct = codec.resample_packed(packed, lengths, o, t, out_lengths=[3000] * len(clips), normalize_peak=True)
    finally:
        del os.environ["DS_RESAMPLE_DIRECT"]
    assert torch.equal(table, direct)


def test_normalise_crop_and_pad_against_oracle():
    clips, o, t = _batch()
    packed, lengths = _packed(clips)
    n_out = [P.resample_length(n, a, b) for n, a, b in zip(lengths, o, t)]
    want = [n + 999 if k % 2 else n - 321 for k, n in enumerate(n_out)]           # zero-pad odd items, crop even ones
    out = codec.resample_packed(packed, lengths, o, t, out_lengths=want, normalize_peak=True)
    assert out.numel() == sum(want)
    for k, (y, a, b, got) in enumerate(zip(clips, o, t, _split(out, want))):
        y64 = y.astype(np.float64)
        ref = P.fix_length(P.resample(y64 / np.abs(y64).max(), a, b), want[k])
        assert crel(got, ref) <= 1e-5, (a, b)
        if k % 2:
            assert not got[n_out[k]:].any()
        assert np.abs(got).max() <= 1.1


def test_batched_items_equal_items_alone():
    clips, o, t = _batch()
    packed, lengths = _packed(clips)
    n_out = [P.resample_length(n, a, b) for n, a, b in zip(lengths, o, t)]
    batch = torch.split(codec.resample_packed(packed, lengths, o, t, normalize_peak=True), n_out)
    again = torch.split(codec.resample_packed(packed, lengths, o, t, normalize_peak=True), n_out)
    for k in range(len(clips)):
        alone = codec.resample_packed(torch.from_numpy(clips[k]).cuda(), [lengths[k]], o[k], t[k], normalize_peak=True)
        assert torch.equal(alone, batch[k]) and torch.equal(again[k], batch[k]), PAIRS[k]


def test_resample_dropin_layouts():
    y = _clip(44100, 44100, 3)
    one = codec.resample(y, 44100, 16000)                                   # [L] numpy -> [n] numpy
    assert isinstance(one, np.ndarray) and one.dtype == np.float32 and one.shape == (16000,)
    two = codec.resample(np.stack([y, y[::-1].copy()]), 44100.0, 16000)     # [B, L] numpy, integral float rate
    assert isinstance(two, np.ndarray) and two.shape == (2, 16000) and np.array_equal(two[0], one)
    dev = codec.resample(torch.from_numpy(y).cuda(), 44100, 16000)          # tensor in, tensor out
    assert dev.is_cuda and torch.equal(dev.cpu(), torch.from_numpy(one))
    z = _clip(48000, 30000, 4)
    parts = codec.resample([y, z], [44100, 48000], 16000)                   # a list with one rate per item
    assert [p.shape for p in parts] == [(16000,), (10000,)] and np.array_equal(parts[0], one)
    assert np.array_equal(parts[1], codec.resample(z, 48000, 16000))
    assert np.array_equal(codec.resample(y, 44100, 44100), y)               # equal rates: the input
    odd = codec.resample(y[:147], 44100, 48000)
    assert odd.shape == (161,)                                              # librosa's float ceil, not ceil-division


def test_resampled_tone_keeps_its_frequency():
    sr, f = 44100, 1234.5
    y = (np.sin(2 * np.pi * f * np.arange(3 * sr) / sr) * 0.8).astype(np.float32)
    z = codec.resample(y, sr, 16000).astype(np.float64)
    peak = np.argmax(np.abs(np.fft.rfft(z * np.hanning(len(z))))) * 16000 / len(z)
    assert abs(peak - f) <= 16000 / len(z)
    t = np.arange(len(z)) / 16000
    s = slice(500, len(z) - 500)
    assert np.abs(z[s] - 0.8 * np.sin(2 * np.pi * f * t[s])).max() < 1e-4


@pytest.fixture(scope="module")
def pipe():
    from diffusynth_b200 import TextToTimbre
    return TextToTimbre.random_init(device="cuda", seed=0, batch_invariant=True)


def _encode_before(pipe, wave, width=64):
    """encode_audio as it was before uploads could have other rates: torch normalisation, adjust_audio_length, STFT, encoder."""
    wave = wave.to(pipe.device, torch.float32)
    wave = wave / wave.abs().amax(dim=-1, keepdim=True).clamp_min(1e-12)
    wave = adjust_audio_length(wave, 256 * (4 * width - 1))
    spec = waveform_to_spectrogram(wave, time_resolution=max(256, 4 * width))
    return pipe.vqgan._encoder(spec)


@pytest.mark.parametrize("L", [65280, 70001, 50000])
def test_encode_audio_16k_is_unchanged(pipe, L):
    wave = torch.from_numpy(np.stack([_clip(16000, L, 60), 0.01 * _clip(16000, L, 61)])).cuda()
    assert torch.equal(pipe.encode_audio(wave), _encode_before(pipe, wave))
    assert torch.equal(pipe.encode_audio(wave[:1], width=48), _encode_before(pipe, wave[:1], width=48))


def test_encode_audio_mixed_rate_uploads(pipe):
    srs = [44100, 48000, 22050, 16000]
    clips = [_clip(sr, int(sr * d), 70 + k) for k, (sr, d) in enumerate(zip(srs, (4.5, 3.2, 4.08, 2.0)))]
    lat = pipe.encode_audio(clips, sample_rate=srs)
    assert tuple(lat.shape) == (4, 4, 128, 64)
    for k in range(len(clips)):
        assert torch.equal(pipe.encode_audio([clips[k]], sample_rate=srs[k]), lat[k:k + 1]), srs[k]
    n = 256 * 255
    packed, lengths = _packed(clips)
    wave = codec.resample_packed(packed, lengths, srs, 16000, out_lengths=n, normalize_peak=True).view(len(clips), n)
    assert torch.equal(pipe.vqgan._encoder(waveform_to_spectrogram(wave)), lat)              # the encoder's input is that wave
    for k, (y, sr) in enumerate(zip(clips, srs)):
        ref_wave, _ = P.upload_chain(y.astype(np.float64), sr)
        e = crel(wave[k].cpu().numpy().astype(np.float64), ref_wave)
        print(f"\nupload at {sr} Hz: encoder input rel-L2 vs oracle chain {e:.2e}")
        assert e <= 1e-5


def _counting(lib):
    class Counting:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            fn = getattr(lib, name)
            if not name.startswith("ds_"):
                return fn

            def wrapped(*a):
                self.calls.append(name)
                return fn(*a)
            return wrapped
    return Counting()


def test_encode_audio_issues_fixed_library_calls(pipe):
    counts = []
    for n_clips in (2, 5):
        srs = [(44100, 48000, 22050)[k % 3] for k in range(n_clips)]
        clips = [_clip(sr, sr * 3 + 100 * k, 80 + k) for k, sr in enumerate(srs)]
        pipe.encode_audio(clips, sample_rate=srs)                    # warm: plans and buffers of this batch size
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            pipe.encode_audio(clips, sample_rate=srs)
        finally:
            _lib._lib = real
        counts.append(sorted(proxy.calls))
    print(f"\nencode_audio library calls: {len(counts[0])} ({counts[0].count('ds_resample')} ds_resample)")
    assert counts[0] == counts[1] and counts[0].count("ds_resample") == 1 and counts[0].count("ds_resample_workspace") == 1


def test_modify_with_uploads_at_two_rates(pipe):
    clips = [_clip(44100, 44100 * 4, 90), _clip(48000, 48000 * 3, 91)]
    guide = pipe.encode_audio(clips, sample_rate=[44100, 48000])
    steps, strength = 3, 0.7
    draws = W.host_noise(12, 1 + int(steps / strength), 2)
    cond, uncond = W.synthetic_conditions(2, 512)
    both = pipe.modify(guide, cond.cuda(), uncond.cuda(), steps=steps, strength=strength, noise_feed=draws).waveforms
    assert torch.isfinite(both).all() and both.abs().max() > 0
    for k in range(2):
        alone = pipe.modify(guide[k:k + 1], cond[k:k + 1].cuda(), uncond.cuda(), steps=steps, strength=strength,
                            noise_feed=draws[:, k:k + 1]).waveforms
        assert torch.equal(alone[0], both[k]), k
