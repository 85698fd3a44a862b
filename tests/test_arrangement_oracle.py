"""Multi-instrument arrangements without a GPU: the float64 arrangement oracle (tests/arrangement_oracle.py) against
pitch_oracle.mix_track and hand-computed envelopes, the host-side plan of TextToTimbre.render_arrangement, and the argument checks
of ds_mix_arrangement, which run before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib
from tests import arrangement_oracle as A
from tests import pitch_oracle as P


def _tracks(notes=A.HAND_NOTES):
    lat, cond = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512)
    return [(lat, cond, n, g, f) for n, g, f in notes]


def test_arrangement_plan_of_the_hand_case():
    from diffusynth_b200.pipeline import TextToTimbre
    p = TextToTimbre.arrangement_plan(_tracks())
    for k, v in A.HAND_PLAN.items():
        assert getattr(p, k) == v, k
    assert p.widths == [TextToTimbre.note_width(d) for _, d in p.rows]


def test_plan_groups_rows_across_tracks_and_pairs_once():
    from diffusynth_b200.pipeline import TextToTimbre
    p = TextToTimbre.arrangement_plan(_tracks())
    groups = {w: [r for r, ww in enumerate(p.widths) if ww == w] for w in p.widths}
    assert groups == {30: [0, 2], 48: [1, 4], 64: [3]}                       # rows of tracks 0/1 and 0/2 share a launch
    assert {p.rows[r][0] for r in groups[30]} == {0, 1} and {p.rows[r][0] for r in groups[48]} == {0, 2}
    assert len(p.items) == len(set(p.items)) == 6 < len(p.note_item) == 8    # (0.9 s, 0) of track 0 and (2.0 s, +5) of track 2 repeat
    assert p.note_item.count(0) == 2 and p.note_item.count(4) == 2
    one = TextToTimbre.track_plan(A.HAND_NOTES[0][0])                         # one track: the rows and items of track_plan
    solo = TextToTimbre.arrangement_plan(_tracks(A.HAND_NOTES[:1]))
    assert [d for _, d in solo.rows] == one.durations and solo.items == one.pairs and solo.note_item == one.note_pair


def test_plan_rejects_bad_arrangements():
    from diffusynth_b200.pipeline import TextToTimbre
    with pytest.raises(ValueError):
        TextToTimbre.arrangement_plan([])
    with pytest.raises(ValueError):
        TextToTimbre.arrangement_plan(_tracks([([], 1.0, 0.0)]))
    for fade in (-0.01, float("nan")):
        with pytest.raises(ValueError):
            TextToTimbre.arrangement_plan(_tracks([([(0.0, 1.0, 0, 1.0)], 1.0, fade)]))


def test_oracle_without_fades_or_peak_is_mix_track():
    rng = np.random.default_rng(4)
    waves = [rng.standard_normal(n) for n in (300, 1000, 45, 700)]
    onsets, gains = [0, 120, 900, 333], [0.5, -1.0, 2.0, 0.75]
    assert np.array_equal(A.mix_arrangement(waves, onsets, gains, [0] * 4), P.mix_track(waves, onsets, gains))


def test_envelope_ramp_ends_and_clamp():
    env = A.envelope(10, 4)
    assert np.array_equal(env[:6], np.ones(6))
    assert env[6] == 1.0 and env[9] == 0.25                                  # (L - i) / F: first ramp sample 4/4, last 1/4
    assert np.allclose(env[6:], [1.0, 0.75, 0.5, 0.25])
    assert np.array_equal(A.envelope(10, 0), np.ones(10))
    long = A.envelope(5, 50)                                                 # a fade longer than its note covers the whole note
    assert np.array_equal(long, A.envelope(5, 5)) and np.allclose(long, [1.0, 0.8, 0.6, 0.4, 0.2])
    tr = A.mix_arrangement([np.ones(4), np.ones(3)], [0, 2], [1.0, 2.0], [2, 1])
    assert np.allclose(tr, [1.0, 1.0, 3.0, 2.5, 2.0])


def test_oracle_peak_normalisation():
    tr = A.mix_arrangement([np.array([0.5, -2.0, 1.0])], [1], [1.0], [0], target_peak=0.9)
    assert np.allclose(tr, [0.0, 0.225, -0.9, 0.45])
    assert not A.mix_arrangement([np.zeros(5)], [0], [1.0], [2], target_peak=0.9).any()


def _arr(vals, ctype):
    return (ctype * len(vals))(*vals)


def test_mix_arrangement_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(0)
    L = C.c_longlong
    lens, on, fades = _arr([100, 50], L), _arr([0, 60], L), _arr([10, 0], L)
    assert lib.ds_mix_arrangement_workspace(lens, on, fades, 2, 0.0, 110, C.byref(nbytes)) == 0
    plain = nbytes.value
    assert lib.ds_mix_arrangement_workspace(lens, on, fades, 2, 0.9, 5000, C.byref(nbytes)) == 0
    assert nbytes.value > plain                                              # + the peak partials
    assert lib.ds_mix_arrangement_workspace(lens, on, _arr([10, -1], L), 2, 0.0, 110, C.byref(nbytes)) == -1
    assert b"fade_out" in lib.ds_last_error()
    for peak in (float("nan"), -0.5, float("inf")):
        assert lib.ds_mix_arrangement_workspace(lens, on, fades, 2, peak, 110, C.byref(nbytes)) == -1
        assert b"target_peak" in lib.ds_last_error()
    assert lib.ds_mix_arrangement_workspace(lens, on, fades, 2, 0.0, 109, C.byref(nbytes)) == -1
    assert b"past the track length" in lib.ds_last_error()
    assert lib.ds_mix_arrangement_workspace(lens, on, None, 2, 0.0, 110, C.byref(nbytes)) == -1
    offs, gains = _arr([0, 100], L), _arr([1.0, 0.5], C.c_float)
    dev = C.c_void_p(16)                                                     # never dereferenced: every check fails first
    assert lib.ds_mix_arrangement(dev, _arr([0, -1], L), lens, on, gains, fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert b"source offset" in lib.ds_last_error()
    assert lib.ds_mix_arrangement(dev, offs, lens, on, gains, _arr([-3, 0], L), 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert lib.ds_mix_arrangement(dev, offs, lens, on, gains, fades, 2, float("nan"), dev, 110, dev, 1 << 40, None) == -1
    assert lib.ds_mix_arrangement(None, offs, lens, on, gains, fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert lib.ds_mix_arrangement(dev, offs, lens, on, gains, fades, 2, 0.0, dev, 110, dev, 8, None) == -1
    assert b"workspace" in lib.ds_last_error()


def test_python_surface_rejects_bad_fades_and_peaks_before_the_device():
    from diffusynth_b200 import codec
    args = (torch.zeros(100), [0], [100], [0], [1.0])
    with pytest.raises(ValueError):
        codec.mix_arrangement(*args, [-1])
    for peak in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            codec.mix_arrangement(*args, [0], target_peak=peak)


def test_render_arrangement_rejects_bad_input_before_synthesis():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def no_synthesis(*a):
        raise AssertionError("synthesis reached")
    pipe._synthesize_rows = no_synthesis
    lat, cond, notes = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512), [(0.0, 1.0, 0, 1.0)]
    bad = [[], [(lat, cond, [], 1.0, 0.0)], [(lat[:, :3], cond, notes, 1.0, 0.0)], [(torch.zeros(2, 4, 128, 64), cond, notes, 1.0, 0.0)],
           [(lat, torch.zeros(512), notes, 1.0, 0.0)], [(lat, cond, notes, 1.0, -0.5)]]
    for tracks in bad:
        with pytest.raises(ValueError):
            pipe.render_arrangement(tracks)
    for peak in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            pipe.render_arrangement([(lat, cond, notes, 1.0, 0.0)], target_peak=peak)


def test_render_track_rejects_bad_input_before_synthesis():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def no_synthesis(*a):
        raise AssertionError("synthesis reached")
    pipe._synthesize_rows = no_synthesis
    lat, cond, notes = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512), [(0.0, 1.0, 0, 1.0)]
    for args in ((lat[:, :3], cond, notes), (lat, torch.zeros(512), notes), (lat, cond, [])):
        with pytest.raises(ValueError):
            pipe.render_track(*args)
