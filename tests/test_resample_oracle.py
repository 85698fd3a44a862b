"""Sample-rate conversion without a GPU: the float64 restatements of librosa.resample(res_type="kaiser_best") in
tests/resample_oracle.py (librosa's output length, the identity at equal rates, the polyphase form the device computes, analytic
resampling of band-limited tones), and the argument checks of ds_resample / ds_resample_workspace, which run before any device
work."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec
from tests import resample_oracle as P

PAIRS = [(8000, 16000), (11025, 16000), (22050, 16000), (32000, 16000), (44100, 16000), (48000, 16000), (96000, 16000),
         (16000, 44100), (16000, 48000), (44101, 16000)]


def test_length_rule_is_librosas_float_ceil():
    assert P.resample_length(147, 44100, 48000) == 161           # integer ceil-division gives 160
    assert P.resample_length(147, 11025, 48000) == 641           # 640
    assert codec.resample_length(147, 44100, 48000) == 161 and codec.resample_length(147, 11025, 48000) == 641
    for n, o, t in ((65280 * 441 // 160, 44100, 16000), (196000, 48000, 16000), (1000, 16000, 44100), (7, 3, 5)):
        assert P.resample_length(n, o, t) == int(np.ceil(n * (float(t) / o))) == codec.resample_length(n, o, t)
        assert len(P.resample(np.ones(n), o, t)) == P.resample_length(n, o, t)


def test_equal_rates_are_the_identity():
    y = np.random.default_rng(1).standard_normal(1234)
    for sr in (16000, 44100):
        assert np.array_equal(P.resample(y, sr, sr), y)
        assert np.array_equal(P.resample_polyphase(y, sr, sr), y)


@pytest.mark.parametrize("o,t", PAIRS)
def test_polyphase_restatement_matches_resample_kaiser(o, t):
    """The phases indexed in integers (base (j*down) div up, phase (j*down) mod up) give resample_kaiser's sum.  resample_kaiser
    decides taps exactly at the support's edge (|d| = 64/s) from float64 positions, the polyphase form in integers, so the two may
    differ there by at most one edge tap per side of an output."""
    y = np.random.default_rng(o + t).standard_normal(6001)
    a, b = P.resample_kaiser(y, float(t) / o), P.resample_polyphase(y, o, t)
    assert len(a) == len(b) == P.resample_length(len(y), o, t)
    tab, up, down, F = P.polyphase_table(o, t)
    assert tab.shape == (up, 2 * F + 2)
    sc = min(1.0, float(t) / o)
    edge = P.RS_ROLLOFF * sc * abs(np.sinc(P.RS_ROLLOFF * P.RS_ZEROS)) / np.i0(P.RS_BETA)       # h at |d| = 64/s
    err = np.abs(a - b).max() / np.abs(a).max()
    print(f"\n{o} -> {t}: up {up}, down {down}, {2 * F + 2} taps, max |polyphase - direct| / max {err:.2e}")
    assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max() + 2 * edge * np.abs(y).max()
    if up == 1 or down == 1:
        assert err <= 1e-12                                    # edges on whole samples: both decide them alike


@pytest.mark.parametrize("o,t", [(8000, 16000), (22050, 16000), (44100, 16000), (48000, 16000), (16000, 44100), (16000, 48000)])
def test_resample_band_limited_tones(o, t):
    f_max = 0.4 * min(o, t)
    sig = lambda x: np.sin(2 * np.pi * 0.31 * f_max * x) + 0.5 * np.sin(2 * np.pi * f_max * x + 1)
    y = sig(np.arange(4 * o // 10) / o)
    r = P.resample_polyphase(y, o, t)
    assert len(r) == P.resample_length(len(y), o, t)
    tt = np.arange(len(r)) / t
    edge = int(0.03 * t)                                       # the filter's reach (64 zero crossings) plus margin
    s = slice(edge, len(r) - edge)
    assert np.abs(r[s] - sig(tt[s])).max() < 1e-5


def test_upload_chain_normalises_then_resamples():
    y = 3.0 * np.sin(2 * np.pi * 440 * np.arange(44100) / 44100)
    wave, spec = P.upload_chain(y, 44100, width=64)
    assert wave.shape == (256 * 255,) and spec.shape == (3, 512, 256)
    assert 0.95 < np.abs(wave[2000:-2000]).max() <= 1.01


def _arr(vals, ctype):
    return (ctype * len(vals))(*vals)


def test_resample_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(0)
    L, o, t = _arr([1000, 2000], C.c_longlong), _arr([44100, 48000], C.c_longlong), _arr([16000, 16000], C.c_longlong)
    assert lib.ds_resample_workspace(L, o, t, None, 2, C.byref(nbytes)) == 0 and nbytes.value > 0
    big = nbytes.value
    assert lib.ds_resample_workspace(L, o, t, _arr([65280, 1], C.c_longlong), 2, C.byref(nbytes)) == 0
    bad = (([1000, 0], [44100, 48000], [16000, 16000], None),                 # non-positive length
           ([1000, -3], [44100, 48000], [16000, 16000], None),
           ([1000, 2000], [44100, 0], [16000, 16000], None),                  # non-positive rate
           ([1000, 2000], [44100, 48000], [16000, -16000], None),
           ([1000, 2000], [44100, 48000], [16000, 4194305], None),           # rate above DS_RESAMPLE_MAX_RATE
           ([1000, 2000], [1 << 40, 48000], [16000, 16000], None),
           ([1000, 2000], [44100, 48000], [16000, 16000], [65280, 0]),        # non-positive output length
           ([(1 << 40) + 1, 2000], [44100, 48000], [16000, 16000], None))     # length above DS_RESAMPLE_MAX_LENGTH
    for lens, si, so, ol in bad:
        args = (_arr(lens, C.c_longlong), _arr(si, C.c_longlong), _arr(so, C.c_longlong), None if ol is None else _arr(ol, C.c_longlong))
        assert lib.ds_resample_workspace(*args, 2, C.byref(nbytes)) == -1
        assert b"ds_resample_workspace" in lib.ds_last_error()
        assert lib.ds_resample(C.c_void_p(16), C.c_void_p(16), *args, 1, 2, C.c_void_p(16), 1 << 40, None) == -1
        assert b"ds_resample" in lib.ds_last_error()
    assert lib.ds_resample_workspace(None, o, t, None, 2, C.byref(nbytes)) == -1
    assert lib.ds_resample_workspace(L, None, t, None, 2, C.byref(nbytes)) == -1
    assert lib.ds_resample_workspace(L, o, None, None, 2, C.byref(nbytes)) == -1
    assert lib.ds_resample_workspace(L, o, t, None, 2, None) == -1
    assert lib.ds_resample_workspace(L, o, t, None, 0, C.byref(nbytes)) == -1
    assert lib.ds_resample_workspace(L, o, t, None, -1, C.byref(nbytes)) == -1
    assert lib.ds_resample(None, C.c_void_p(16), L, o, t, None, 0, 2, C.c_void_p(16), big, None) == -1
    assert lib.ds_resample(C.c_void_p(16), None, L, o, t, None, 0, 2, C.c_void_p(16), big, None) == -1
    assert lib.ds_resample(C.c_void_p(16), C.c_void_p(16), L, o, t, None, 0, 2, None, big, None) == -1
    assert lib.ds_resample(C.c_void_p(16), C.c_void_p(16), L, o, t, None, 0, 0, C.c_void_p(16), big, None) == -1
    assert lib.ds_resample(C.c_void_p(16), C.c_void_p(16), L, o, t, None, 0, 2, C.c_void_p(16), big - 1, None) == -1
    assert b"workspace" in lib.ds_last_error()


def test_python_surface_rejects_bad_rates_and_layouts_before_the_device():
    for bad in (16000.5, 0, -8000, float("nan"), "16000", None, 1 << 23):
        with pytest.raises(ValueError):
            codec.resample_packed(torch.zeros(100), [100], bad, 16000)
        with pytest.raises(ValueError):
            codec.resample(np.zeros(100, np.float32), 44100, bad)
    with pytest.raises(ValueError):
        codec.resample(np.zeros((2, 3, 100), np.float32), 44100, 16000)
    with pytest.raises(ValueError):
        codec.resample([np.zeros(100, np.float32), np.zeros((2, 50), np.float32)], 44100, 16000)
    with pytest.raises(ValueError):
        codec.resample(np.zeros((2, 100), np.float32), [44100, 48000], 16000)      # rows would differ in length
