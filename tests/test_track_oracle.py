"""Note arrangements without a GPU: the float64 restatements of librosa.effects.pitch_shift's pieces (tests/pitch_oracle.py)
against torch and analytic results, the host-side track plan of TextToTimbre.render_track, and the argument checks of the
pitch-shift / mix entry points, which run before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib
from oracle import ds_oracle as O
from tests import pitch_oracle as P

SR = 16000


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def decaying_tone(L, f=440.0):
    t = np.arange(L) / SR
    return np.sin(2 * np.pi * f * t) * np.exp(-t)


@pytest.mark.parametrize("L", [30464, 48896, 5000])
def test_stft_istft_2048_match_torch(L):
    y = np.random.default_rng(L).standard_normal(L)
    D = O.stft(y, n_fft=2048, hop=512)
    win = torch.hann_window(2048, periodic=True, dtype=torch.float64)
    Dt = torch.stft(torch.from_numpy(y), 2048, 512, 2048, win, center=True, pad_mode="constant", return_complex=True).numpy()
    assert D.shape == (1025, 1 + L // 512)
    assert np.abs(D - Dt).max() <= 1e-12 * np.abs(Dt).max()
    for length in (L, L - 700, int(round(L * 1.3))):
        S = D if length <= L else P.phase_vocoder(D, L / length)       # a longer spectrum for the longer length
        ref = torch.istft(torch.from_numpy(S), 2048, 512, 2048, win, center=True, length=length).numpy()
        got = P.istft_length(S, 512, length)
        assert got.shape == (length,)
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max(), length


def test_istft_length_at_the_natural_length_is_istft():
    D = O.stft(np.random.default_rng(3).standard_normal(12000), n_fft=2048, hop=512)
    ref = O.istft(D, hop=512, win=2048)
    assert np.array_equal(P.istft_length(D, 512, len(ref)), ref)


def test_pitch_shift_zero_is_identity():
    y = decaying_tone(30464) + 0.1 * np.random.default_rng(0).standard_normal(30464)
    D = O.stft(y, 2048, 512)
    assert rel(P.phase_vocoder(D, 1.0), D) < 1e-10       # at rate 1 the vocoder reproduces D (its phase grows to ~1e4 rad)
    assert rel(P.pitch_shift(y, 0), y) < 1e-10


@pytest.mark.parametrize("n", [-12, -7, 5, 12])
def test_pitch_shift_moves_a_tone(n):
    L = 48896
    z = P.pitch_shift(decaying_tone(L), n)
    assert z.shape == (L,)
    F = np.abs(np.fft.rfft(z * np.hanning(L)))
    peak = np.argmax(F) * SR / L
    assert abs(peak - 440.0 * 2 ** (n / 12)) <= SR / L, (peak, 440.0 * 2 ** (n / 12))


@pytest.mark.parametrize("ratio", [2 ** (-7 / 12), 2 ** (7 / 12)])
def test_resampler_matches_analytic_resampling(ratio):
    sig = lambda t: np.sin(2 * np.pi * 1234.5 * t) + 0.5 * np.sin(2 * np.pi * 3100 * t + 1)       # band-limited below both Nyquists
    x = sig(np.arange(20000) / SR)
    r = P.resample_kaiser(x, ratio)
    assert len(r) == int(np.ceil(20000 * ratio))
    t = np.arange(len(r)) / (SR * ratio)
    s = slice(500, len(r) - 500)
    assert np.abs(r[s] - sig(t[s])).max() < 1e-6


def test_mix_track_oracle():
    w = [np.arange(5.0), np.ones(3), -np.ones(4)]
    tr = P.mix_track(w, [0, 2, 7], [1.0, 0.5, 2.0])
    assert tr.shape == (11,)
    assert np.allclose(tr, [0, 1, 2.5, 3.5, 4.5, 0, 0, -2, -2, -2, -2])


def test_track_plan_groups_notes():
    from diffusynth_b200.pipeline import TextToTimbre
    notes = [(0.0, 0.9, 0, 1.0), (0.5, 2.0, -3, 0.5), (1.00003, 0.9, 0, 0.7), (1.25, 0.9, 5, 1.0), (2.0, 3.0, 12, 0.25),
             (2.1, 2.0, -3, 1.0)]
    p = TextToTimbre.track_plan(notes)
    assert p.durations == [0.9, 2.0, 3.0]
    assert p.pairs == [(0, 0.0), (1, -3.0), (0, 5.0), (2, 12.0)]
    assert p.note_pair == [0, 1, 0, 2, 3, 1]
    assert p.onsets == [0, 8000, 16000, 20000, 32000, 33600]
    assert p.gains == [1.0, 0.5, 0.7, 1.0, 0.25, 1.0]
    widths = [TextToTimbre.note_width(d) for _, d, _, _ in notes]
    assert widths == [30, 48, 30, 30, 64, 48]
    assert p.lengths == [256 * (4 * w - 1) for w in widths]
    assert p.track_len == max(o + n for o, n in zip(p.onsets, p.lengths)) == 32000 + 256 * 255
    with pytest.raises(ValueError):
        TextToTimbre.track_plan([(-0.1, 1.0, 0, 1.0)])


def _arr(vals, ctype):
    return (ctype * len(vals))(*vals)


def test_pitch_and_mix_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(0)
    ok_len, ok_steps = _arr([30464, 48896], C.c_longlong), _arr([0.0, -7.0], C.c_double)
    assert lib.ds_pitch_shift_workspace(ok_len, ok_steps, 2, C.byref(nbytes), None) == 0 and nbytes.value > 0
    for lens, steps in (([30464, 0], [0.0, 1.0]), ([30464, -5], [0.0, 1.0]), ([100, 100], [0.0, 24.5]), ([100, 100], [-25.0, 0.0]),
                        ([100, 100], [float("nan"), 0.0]), ([100, 100], [float("inf"), 0.0])):
        assert lib.ds_pitch_shift_workspace(_arr(lens, C.c_longlong), _arr(steps, C.c_double), 2, C.byref(nbytes), None) == -1
        assert lib.ds_pitch_shift(C.c_void_p(16), C.c_void_p(16), _arr(lens, C.c_longlong), _arr(steps, C.c_double), 2, C.c_void_p(16),
                                  1 << 40, None) == -1
        assert b"ds_pitch_shift" in lib.ds_last_error()
    assert lib.ds_pitch_shift_workspace(None, ok_steps, 2, C.byref(nbytes), None) == -1
    assert lib.ds_pitch_shift_workspace(ok_len, ok_steps, 0, C.byref(nbytes), None) == -1
    assert lib.ds_pitch_shift(None, C.c_void_p(16), ok_len, ok_steps, 2, C.c_void_p(16), 1 << 40, None) == -1
    assert lib.ds_pitch_shift(C.c_void_p(16), C.c_void_p(16), ok_len, ok_steps, 2, None, 1 << 40, None) == -1
    assert lib.ds_pitch_shift(C.c_void_p(16), C.c_void_p(16), ok_len, ok_steps, 2, C.c_void_p(16), 16, None) == -1    # workspace short
    assert b"workspace" in lib.ds_last_error()

    lens, on = _arr([100, 50], C.c_longlong), _arr([0, 60], C.c_longlong)
    offs, gains = _arr([0, 100], C.c_longlong), _arr([1.0, 0.5], C.c_float)
    assert lib.ds_mix_track_workspace(lens, on, 2, 110, C.byref(nbytes)) == 0 and nbytes.value > 0
    assert lib.ds_mix_track_workspace(lens, on, 2, 109, C.byref(nbytes)) == -1                  # the second note ends at 110
    assert b"past the track length" in lib.ds_last_error()
    assert lib.ds_mix_track_workspace(_arr([100, 0], C.c_longlong), on, 2, 110, C.byref(nbytes)) == -1
    assert lib.ds_mix_track_workspace(lens, _arr([0, -1], C.c_longlong), 2, 110, C.byref(nbytes)) == -1
    assert lib.ds_mix_track(C.c_void_p(16), offs, lens, on, gains, 2, C.c_void_p(16), 109, C.c_void_p(16), 1 << 40, None) == -1
    assert lib.ds_mix_track(None, offs, lens, on, gains, 2, C.c_void_p(16), 110, C.c_void_p(16), 1 << 40, None) == -1
    assert lib.ds_mix_track(C.c_void_p(16), None, lens, on, gains, 2, C.c_void_p(16), 110, C.c_void_p(16), 1 << 40, None) == -1
    assert lib.ds_mix_track(C.c_void_p(16), offs, lens, on, gains, 2, C.c_void_p(16), 110, C.c_void_p(16), 8, None) == -1


def test_python_surface_rejects_bad_steps_before_the_device():
    from diffusynth_b200 import codec
    for bad in (24.01, -30, float("nan")):
        with pytest.raises(ValueError):
            codec.pitch_shift_packed(torch.zeros(100), [100], [bad])
