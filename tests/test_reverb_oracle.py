"""Convolution reverb without a GPU: the mode -> (start, length) rule of codec.fftconvolve against scipy and numpy, the float64
reverb oracle (tests/reverb_oracle.py), the per-note sends of TextToTimbre.arrangement_plan, and the argument checks of
ds_fftconvolve, codec.fftconvolve and render_arrangement's reverb, which all run before any device work."""
import ctypes as C

import numpy as np
import pytest
import scipy.signal
import torch

from diffusynth_b200 import _lib, codec
from tests import arrangement_oracle as A
from tests import reverb_oracle as RV
from tests import stereo_oracle as S

SIZES = (1, 2, 1023, 1024, 1025, 3000)


@pytest.mark.parametrize("mode", codec.CONV_MODES)
def test_mode_range_matches_scipy_and_numpy(mode):
    for n in SIZES:
        for m in SIZES:
            x = np.random.default_rng(n * 7 + m).standard_normal(n)
            h = np.random.default_rng(n + 11 * m).standard_normal(m)
            start, length = codec.fftconvolve_range(n, m, mode)
            ref = scipy.signal.fftconvolve(x, h, mode=mode)
            assert length == len(ref), (n, m)
            if mode != "same":                          # numpy's "same" has max(n, m) samples, scipy's n
                assert length == len(np.convolve(x, h, mode=mode)), (n, m)
            full = np.convolve(x, h, mode="full")
            assert 0 <= start and start + length <= n + m - 1
            np.testing.assert_allclose(full[start:start + length], ref, rtol=0, atol=1e-9 * max(1.0, np.abs(full).max()))
    with pytest.raises(ValueError):
        codec.fftconvolve_range(10, 3, "circular")


def _notes(seed=4):
    rng = np.random.default_rng(seed)
    waves = [rng.standard_normal(n) for n in (300, 1000, 45, 700)]
    return waves, [0, 120, 900, 333], [0.5, -1.0, 2.0, 0.75], [0, 40, 45, 1000]


def test_zero_sends_give_the_dry_oracle_zero_extended():
    waves, onsets, gains, fades = _notes()
    ir = np.random.default_rng(1).standard_normal(1500)
    for peak in (None, 0.8):
        mono = RV.reverb_mix(waves, onsets, gains, fades, [0.0] * 4, ir, target_peak=peak)
        dry = A.mix_arrangement(waves, onsets, gains, fades, target_peak=peak)
        assert mono.shape == (1120 + 1499,) and np.array_equal(mono[:1120], dry) and not mono[1120:].any()
        pans = [-0.8, 0.3, 1.0, -0.1]
        st = RV.reverb_mix(waves, onsets, gains, fades, [0.0] * 4, np.stack([ir, -ir]), pans, target_peak=peak)
        dry = S.mix_stereo(waves, onsets, gains, pans, fades, target_peak=peak)
        assert st.shape == (2, 1120 + 1499) and np.array_equal(st[:, :1120], dry) and not st[:, 1120:].any()


def test_reverb_oracle_wet_path_and_one_peak_for_both_channels():
    waves, onsets, gains, fades = _notes(5)
    pans, sends = [-0.8, 0.3, 1.0, -0.1], [0.2, 0.5, 0.0, 1.0]
    ir = np.random.default_rng(2).standard_normal((2, 900))
    raw = RV.reverb_mix(waves, onsets, gains, fades, sends, ir, pans)
    bus = S.mix_stereo(waves, onsets, [g * s for g, s in zip(gains, sends)], pans, fades)
    dry = S.mix_stereo(waves, onsets, gains, pans, fades, track_len=1120 + 899)
    for c in (0, 1):
        assert np.allclose(raw[c], dry[c] + np.convolve(bus[c], ir[c]), rtol=0, atol=1e-10)
    out = RV.reverb_mix(waves, onsets, gains, fades, sends, ir, pans, target_peak=0.9)
    assert np.isclose(np.abs(out).max(), 0.9, rtol=1e-15)
    assert np.allclose(out, raw * (0.9 / np.abs(raw).max()), rtol=1e-15, atol=0)
    # a mono IR on a stereo piece convolves both channels with it
    one = RV.reverb_mix(waves, onsets, gains, fades, sends, ir[0], pans)
    assert np.allclose(one[1], dry[1] + np.convolve(bus[1], ir[0]), rtol=0, atol=1e-10)


def test_arrangement_plan_carries_track_sends():
    from diffusynth_b200.pipeline import ArrangementPlan, TextToTimbre
    lat, cond = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512)
    tracks = [(lat, cond, n, g, f) for n, g, f in A.HAND_NOTES]
    p = TextToTimbre.arrangement_plan(tracks, reverb_sends=[0.2, 0.0, 1.5])
    for k, v in A.HAND_PLAN.items():
        assert getattr(p, k) == v, k
    assert p.sends == [0.2] * 3 + [0.0] * 2 + [1.5] * 3
    assert TextToTimbre.arrangement_plan(tracks).sends == [1.0] * 8
    for bad in ([0.5, 0.5], [0.1, -0.1, 0.0], [0.0, float("nan"), 0.0], [float("inf"), 0.0, 0.0]):
        with pytest.raises(ValueError, match="reverb_sends"):
            TextToTimbre.arrangement_plan(tracks, reverb_sends=bad)
    # existing positional constructions still work: sends default to empty like pans
    plan = ArrangementPlan([], [], [], [], [], [], [], [], 0)
    assert plan.pans == [] and plan.sends == []


def _arr(vals, ctype):
    return (ctype * len(vals))(*vals)


L = C.c_longlong


def test_fftconvolve_argument_errors_without_gpu():
    lib = _lib.load()
    b = L(0)
    xl, hl, hi, st, ol = _arr([100, 2000], L), _arr([50], L), _arr([0, 0], L), _arr([0, 10], L), _arr([149, 2039], L)
    ws = lib.ds_fftconvolve_workspace
    assert ws(xl, 2, hl, 1, hi, st, ol, 0.0, C.byref(b)) == 0
    plain = b.value
    # 24 int64 of metadata, the spectra of 1 + 2 blocks and 1 partition, segment 0 of item 0 and segments 0..1 of item 1 (its
    # full convolution has 2 segments), each 256-byte aligned
    assert plain == 256 + 33024 + 3 * 2048 * 4
    assert ws(xl, 2, hl, 1, hi, st, ol, 0.9, C.byref(b)) == 0 and b.value > plain          # + the peak partials
    cases = [
        ((None, 2, hl, 1, hi, st, ol, 0.0), b"must be non-null"),
        ((xl, 2, None, 1, hi, st, ol, 0.0), b"must be non-null"),
        ((xl, 2, hl, 1, None, st, ol, 0.0), b"must be non-null"),
        ((xl, 2, hl, 1, hi, None, ol, 0.0), b"must be non-null"),
        ((xl, 2, hl, 1, hi, st, None, 0.0), b"must be non-null"),
        ((xl, 0, hl, 1, hi, st, ol, 0.0), b"B = 0"),
        ((xl, 2, hl, 0, hi, st, ol, 0.0), b"H = 0"),
        ((_arr([100, 0], L), 2, hl, 1, hi, st, ol, 0.0), b"item 1 has length 0"),
        ((xl, 2, _arr([0], L), 1, hi, st, ol, 0.0), b"impulse response 0 has length 0"),
        ((xl, 2, hl, 1, _arr([0, 1], L), st, ol, 0.0), b"item 1 has h_index 1"),
        ((xl, 2, hl, 1, _arr([-1, 0], L), st, ol, 0.0), b"item 0 has h_index -1"),
        ((xl, 2, hl, 1, hi, _arr([0, -1], L), ol, 0.0), b"out_start -1"),
        ((xl, 2, hl, 1, hi, st, _arr([149, 0], L), 0.0), b"out_length 0"),
        ((xl, 2, hl, 1, hi, st, _arr([150, 2039], L), 0.0), b"past its full length 149"),
        ((xl, 2, hl, 1, hi, _arr([0, 11], L), ol, 0.0), b"past its full length 2049"),
        ((xl, 2, hl, 1, hi, st, ol, float("nan")), b"target_peak"),
        ((xl, 2, hl, 1, hi, st, ol, float("inf")), b"target_peak"),
        ((xl, 2, hl, 1, hi, st, ol, -0.5), b"target_peak"),
    ]
    for args, msg in cases:
        assert ws(*args, C.byref(b)) == -1
        err = lib.ds_last_error()
        assert b"ds_fftconvolve_workspace" in err and msg in err, (err, msg)
    assert ws(xl, 2, hl, 1, hi, st, ol, 0.0, None) == -1
    dev = C.c_void_p(16)                                                     # never dereferenced: every check fails first
    run = lib.ds_fftconvolve
    for args, msg in cases:
        assert run(dev, dev, dev, *args[:7], 0, args[7], dev, 1 << 40, None) == -1
        err = lib.ds_last_error()
        assert b"ds_fftconvolve:" in err and msg in err, (err, msg)
    for null in range(4):
        ptrs = [dev, dev, dev, dev]
        ptrs[null] = None
        assert run(ptrs[0], ptrs[1], ptrs[2], xl, 2, hl, 1, hi, st, ol, 0, 0.0, ptrs[3], 1 << 40, None) == -1
        assert b"must be non-null" in lib.ds_last_error()
    assert run(dev, dev, dev, xl, 2, hl, 1, hi, st, ol, 2, 0.0, dev, 1 << 40, None) == -1
    assert b"accumulate" in lib.ds_last_error()
    assert run(dev, dev, dev, xl, 2, hl, 1, hi, st, ol, 0, 0.0, dev, plain - 1, None) == -1
    assert b"ds_fftconvolve: workspace" in lib.ds_last_error()


def test_codec_fftconvolve_rejects_before_the_device():
    x, h = np.ones(100, dtype=np.float32), np.ones(10, dtype=np.float32)
    for axes in (0, 1, None, (0,), [-1, 0]):
        with pytest.raises(NotImplementedError):
            codec.fftconvolve(x, h, axes=axes)
    with pytest.raises(NotImplementedError):
        codec.fftconvolve(np.ones((2, 3, 100)), h)
    with pytest.raises(NotImplementedError):
        codec.fftconvolve([np.ones((2, 100))], h)
    with pytest.raises(NotImplementedError):
        codec.fftconvolve(x.astype(np.complex64), h)
    with pytest.raises(NotImplementedError):
        codec.fftconvolve(x, torch.ones(10, dtype=torch.complex64))
    for a, b in ((np.ones(0), h), (x, np.ones(0)), (np.ones((0, 5)), h), ([x, np.ones(0)], h), ([], h), (np.float32(1.0), h)):
        with pytest.raises(ValueError):
            codec.fftconvolve(a, b)
    with pytest.raises(ValueError, match="mode"):
        codec.fftconvolve(x, h, mode="circular")
    with pytest.raises(ValueError, match="one per item"):
        codec.fftconvolve([x, x, x], [h, h])
    with pytest.raises(ValueError, match="same output length"):
        codec.fftconvolve(np.ones((2, 100)), [h, np.ones(20)])
    xs = torch.ones(100)
    with pytest.raises(ValueError, match="h_index"):
        codec.fftconvolve_packed(xs, [100], torch.ones(10), [10], h_index=[1])
    with pytest.raises(ValueError, match="accumulate"):
        codec.fftconvolve_packed(xs, [100], torch.ones(10), [10], accumulate=True)
    for peak in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError, match="target_peak"):
            codec.fftconvolve_packed(xs, [100], torch.ones(10), [10], target_peak=peak)


def test_render_arrangement_rejects_bad_reverb_before_synthesis():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def no_synthesis(*a):
        raise AssertionError("synthesis reached")
    pipe._synthesize_rows = no_synthesis
    lat, cond, notes = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512), [(0.0, 1.0, 0, 1.0)]
    tracks = [(lat, cond, notes, 1.0, 0.0), (lat, cond, notes, 0.5, 0.0)]
    ir = np.ones(100)
    with pytest.raises(ValueError, match="stereo=True"):
        pipe.render_arrangement(tracks, impulse_response=np.ones((2, 100)))
    for bad in (np.ones((3, 100)), np.ones((1, 100)), np.ones((2, 2, 100)), np.float64(1.0), np.ones(0), np.ones((2, 0)),
                np.array([1.0, np.nan]), np.array([np.inf, 0.0]), np.array([1e300]), np.ones(5, dtype=np.complex64)):
        with pytest.raises(ValueError, match="impulse_response"):
            pipe.render_arrangement(tracks, impulse_response=bad, stereo=True)
    with pytest.raises(ValueError, match="impulse_response"):
        pipe.render_arrangement(tracks, reverb_sends=[0.5, 0.5])
    for sends in ([0.5], [0.5, 0.5, 0.5], [0.5, -0.1], [float("nan"), 0.0], [0.0, float("inf")]):
        with pytest.raises(ValueError, match="reverb_sends"):
            pipe.render_arrangement(tracks, impulse_response=ir, reverb_sends=sends)
        with pytest.raises(ValueError, match="reverb_sends"):
            pipe.render_arrangement(tracks, impulse_response=torch.ones(2, 100), reverb_sends=sends, stereo=True)
    with pytest.raises(ValueError, match="target_peak"):
        pipe.render_arrangement(tracks, impulse_response=ir, target_peak=float("nan"))
