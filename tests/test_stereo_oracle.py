"""Stereo arrangements without a GPU: the float64 stereo oracle (tests/stereo_oracle.py) -- its pan law and its reduction to the
mono arrangement oracle -- the per-note pans of TextToTimbre.arrangement_plan, the argument checks of ds_mix_stereo, which run
before any device work, and the workspace sizes of the mono mixes, which stereo leaves as they were."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib
from tests import arrangement_oracle as A
from tests import stereo_oracle as S


def test_pan_law_endpoints_centre_swap_and_power():
    for g in (1.0, 0.37, -2.5):
        assert S.pan_gains(g, -1.0) == (g, 0.0)                              # hard left: exact gain, nothing on the right
        assert S.pan_gains(g, 1.0) == (0.0, g)
        left, right = S.pan_gains(g, 0.0)
        assert left == right and np.isclose(left, g / np.sqrt(2.0), rtol=1e-15, atol=0)   # -3 dB each
        for p in (0.1, 0.5, 0.77, 1.0, 1e-7, np.float32(0.3)):
            l1, r1 = S.pan_gains(g, p)
            l2, r2 = S.pan_gains(g, -p)
            assert (l1, r1) == (r2, l2)                                      # mirrored pans swap the gains exactly
            assert np.isclose(l1 * l1 + r1 * r1, g * g, rtol=1e-15, atol=0)  # constant power
            assert S.pan_gains(g, p, fp32=True)[::-1] == S.pan_gains(g, -p, fp32=True)
    assert S.pan_cos(2.0) == 0.0 and np.cos(np.pi / 2) != 0.0


def _notes(seed=4):
    rng = np.random.default_rng(seed)
    waves = [rng.standard_normal(n) for n in (300, 1000, 45, 700)]
    return waves, [0, 120, 900, 333], [0.5, -1.0, 2.0, 0.75], [0, 40, 45, 1000]


def test_hard_left_is_the_mono_arrangement_oracle():
    waves, onsets, gains, fades = _notes()
    for peak in (None, 0.8):
        st = S.mix_stereo(waves, onsets, gains, [-1.0] * 4, fades, target_peak=peak)
        assert st.shape == (2, 1120)
        assert np.array_equal(st[0], A.mix_arrangement(waves, onsets, gains, fades, target_peak=peak))
        assert not st[1].any()
        right = S.mix_stereo(waves, onsets, gains, [1.0] * 4, fades, target_peak=peak)
        assert np.array_equal(right[::-1], st)


def test_stereo_oracle_shares_one_peak_scale():
    waves, onsets, gains, fades = _notes(5)
    pans = [-0.8, 0.3, 1.0, -0.1]
    raw = S.mix_stereo(waves, onsets, gains, pans, fades)
    out = S.mix_stereo(waves, onsets, gains, pans, fades, target_peak=0.9)
    assert np.isclose(np.abs(out).max(), 0.9, rtol=1e-15)
    assert np.allclose(out, raw * (0.9 / np.abs(raw).max()), rtol=1e-15, atol=0)
    assert not S.mix_stereo([np.zeros(5)], [0], [1.0], [0.2], [2], target_peak=0.9).any()


def test_arrangement_plan_carries_track_pans():
    from diffusynth_b200.pipeline import TextToTimbre
    lat, cond = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512)
    pans = [-1.0, 0.25, None]
    tracks = [(lat, cond, n, g, f) + (() if p is None else (p,)) for (n, g, f), p in zip(A.HAND_NOTES, pans)]
    p = TextToTimbre.arrangement_plan(tracks)
    for k, v in A.HAND_PLAN.items():
        assert getattr(p, k) == v, k
    assert p.pans == [-1.0] * 3 + [0.25] * 2 + [0.0] * 3
    assert TextToTimbre.arrangement_plan([t[:5] for t in tracks]).pans == [0.0] * 8
    for bad in (1.5, -1.01, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            TextToTimbre.arrangement_plan([(lat, cond, A.HAND_NOTES[0][0], 1.0, 0.0, bad)])
    with pytest.raises(ValueError):
        TextToTimbre.arrangement_plan([(lat, cond, A.HAND_NOTES[0][0], 1.0, 0.0, 0.0, 0.0)])


def _arr(vals, ctype):
    return (ctype * len(vals))(*vals)


L = C.c_longlong
# (lengths, onsets, fades, track_len) -> ds_mix_track_workspace, then ds_mix_arrangement_workspace at target_peak 0 and 0.9, as the
# library returned them before stereo mixing was added
MONO_WORKSPACES = [
    (([100, 50], [0, 60], [10, 0], 110), (256, 256, 512)),
    (([3000, 4000, 1000], [0, 2500, 5000], [100, 0, 5000], 7000), (256, 256, 512)),
    (([30464] * 7, [0, 1023, 5000, 40000, 90000, 150000, 200000], [0, 9, 30464, 99999, 1, 0, 17], 230464), (2048, 2048, 3072)),
]


@pytest.mark.parametrize("case,expected", MONO_WORKSPACES)
def test_mono_workspace_sizes_are_unchanged(case, expected):
    lib = _lib.load()
    lens, on, fades, tl = case
    b = L(0)
    assert lib.ds_mix_track_workspace(_arr(lens, L), _arr(on, L), len(lens), tl, C.byref(b)) == 0
    got = [b.value]
    for peak in (0.0, 0.9):
        assert lib.ds_mix_arrangement_workspace(_arr(lens, L), _arr(on, L), _arr(fades, L), len(lens), peak, tl, C.byref(b)) == 0
        got.append(b.value)
    assert tuple(got) == expected
    pans = _arr([0.0] * len(lens), C.c_float)
    assert lib.ds_mix_stereo_workspace(_arr(lens, L), _arr(on, L), _arr(fades, L), pans, len(lens), 0.0, tl, C.byref(b)) == 0
    assert b.value >= expected[1]                                            # the float2 gains replace the fp32 ones


def test_mix_stereo_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(0)
    lens, on, fades = _arr([100, 50], L), _arr([0, 60], L), _arr([10, 0], L)
    pans = _arr([-1.0, 0.5], C.c_float)
    assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 2, 0.0, 110, C.byref(nbytes)) == 0
    plain = nbytes.value
    assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 2, 0.9, 5000, C.byref(nbytes)) == 0
    assert nbytes.value > plain                                              # + the peak partials
    for bad in (float("nan"), float("inf"), float("-inf"), 1.001, -2.0):
        assert lib.ds_mix_stereo_workspace(lens, on, fades, _arr([0.0, bad], C.c_float), 2, 0.0, 110, C.byref(nbytes)) == -1
        err = lib.ds_last_error()
        assert b"ds_mix_stereo_workspace" in err and b"note 1 has pan" in err
    assert lib.ds_mix_stereo_workspace(lens, on, fades, None, 2, 0.0, 110, C.byref(nbytes)) == -1
    assert b"pans" in lib.ds_last_error()
    # every check of ds_mix_arrangement_workspace
    assert lib.ds_mix_stereo_workspace(lens, on, _arr([10, -1], L), pans, 2, 0.0, 110, C.byref(nbytes)) == -1
    assert b"fade_out" in lib.ds_last_error()
    for peak in (float("nan"), -0.5, float("inf")):
        assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 2, peak, 110, C.byref(nbytes)) == -1
        assert b"target_peak" in lib.ds_last_error()
    assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 2, 0.0, 109, C.byref(nbytes)) == -1
    assert b"past the track length" in lib.ds_last_error()
    assert lib.ds_mix_stereo_workspace(lens, _arr([0, -1], L), fades, pans, 2, 0.0, 110, C.byref(nbytes)) == -1
    assert b"onset" in lib.ds_last_error()
    assert lib.ds_mix_stereo_workspace(_arr([100, 0], L), on, fades, pans, 2, 0.0, 110, C.byref(nbytes)) == -1
    assert b"length" in lib.ds_last_error()
    assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 0, 0.0, 110, C.byref(nbytes)) == -1
    assert lib.ds_mix_stereo_workspace(lens, on, None, pans, 2, 0.0, 110, C.byref(nbytes)) == -1
    assert lib.ds_mix_stereo_workspace(lens, on, fades, pans, 2, 0.0, 110, None) == -1
    offs, gains = _arr([0, 100], L), _arr([1.0, 0.5], C.c_float)
    dev = C.c_void_p(16)                                                     # never dereferenced: every check fails first
    run = lib.ds_mix_stereo
    assert run(dev, offs, lens, on, gains, _arr([0.0, float("nan")], C.c_float), fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert b"ds_mix_stereo:" in lib.ds_last_error() and b"pan" in lib.ds_last_error()
    assert run(dev, offs, lens, on, gains, _arr([1.5, 0.0], C.c_float), fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, None, fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert b"pans" in lib.ds_last_error()
    assert run(dev, _arr([0, -1], L), lens, on, gains, pans, fades, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert b"source offset" in lib.ds_last_error()
    assert run(dev, offs, lens, on, gains, pans, _arr([-3, 0], L), 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, pans, fades, 2, float("nan"), dev, 110, dev, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, pans, fades, 2, 0.0, dev, 109, dev, 1 << 40, None) == -1
    for null in range(4):
        args = [dev, offs, gains, dev]
        args[null] = None
        assert run(args[0], args[1], lens, on, args[2], pans, fades, 2, 0.0, args[3], 110, dev, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, pans, fades, 2, 0.0, dev, 110, None, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, pans, None, 2, 0.0, dev, 110, dev, 1 << 40, None) == -1
    assert run(dev, offs, lens, on, gains, pans, fades, 2, 0.0, dev, 110, dev, 8, None) == -1
    assert b"ds_mix_stereo: workspace" in lib.ds_last_error()


def test_python_surface_rejects_bad_pans_before_the_device():
    from diffusynth_b200 import codec
    args = (torch.zeros(100), [0], [100], [0], [1.0])
    for pans in ([float("nan")], [float("inf")], [1.5], [-1.01], [0.0, 0.0], []):
        with pytest.raises(ValueError):
            codec.mix_stereo(*args, pans)
    with pytest.raises(ValueError):
        codec.mix_stereo(*args, [0.0], fade_out=[-1])
    for peak in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            codec.mix_stereo(*args, [0.0], target_peak=peak)


def test_render_arrangement_rejects_bad_pans_before_synthesis():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def no_synthesis(*a):
        raise AssertionError("synthesis reached")
    pipe._synthesize_rows = no_synthesis
    lat, cond, notes = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512), [(0.0, 1.0, 0, 1.0)]
    with pytest.raises(ValueError, match="stereo=True"):
        pipe.render_arrangement([(lat, cond, notes, 1.0, 0.0, -1.0)])
    with pytest.raises(ValueError, match="stereo=True"):
        pipe.render_arrangement([(lat, cond, notes, 1.0, 0.0), (lat, cond, notes, 1.0, 0.0, 0.0)])
    for pan in (float("nan"), float("-inf"), 1.0001, -3.0):
        with pytest.raises(ValueError, match="pan"):
            pipe.render_arrangement([(lat, cond, notes, 1.0, 0.0, pan)], stereo=True)
    for tracks in ([], [(lat, cond, notes, 1.0)], [(lat, cond, notes, 1.0, -0.5, 0.0)], [(lat[:, :3], cond, notes, 1.0, 0.0, 0.0)]):
        with pytest.raises(ValueError):
            pipe.render_arrangement(tracks, stereo=True)
    with pytest.raises(ValueError):
        pipe.render_arrangement([(lat, cond, notes, 1.0, 0.0, 0.5)], target_peak=float("nan"), stereo=True)
