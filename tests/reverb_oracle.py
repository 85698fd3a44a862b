"""CPU oracle of convolution reverb on arrangements (TEST INFRASTRUCTURE ONLY): float64 restatements of what
TextToTimbre.render_arrangement(impulse_response=...) computes after synthesis, on top of tests/arrangement_oracle.py and
tests/stereo_oracle.py, with scipy.signal.fftconvolve (float64) as the convolution.

What is assumed (the reference has no reverb): the send is post-fader and post-pan -- the send bus is every note with its gain times
its track's send, the same fades and, in stereo, the same pans -- and the piece is dry + IR * bus, L + M - 1 samples long, the dry
mix zero past L.  A mono IR convolves every channel; a [2, M] IR convolves left with left and right with right.  The peak
normalisation, one factor over both channels, comes after the wet signal is added."""
from __future__ import annotations

import numpy as np
from scipy.signal import fftconvolve

from tests import arrangement_oracle as A
from tests import pitch_oracle as P
from tests import stereo_oracle as S


def reverb_mix(waves, onsets, gains, fades, sends, ir, pans=None, target_peak=None) -> np.ndarray:
    """[L + M - 1] (pans None) or [2, L + M - 1]: the dry mix (arrangement or stereo oracle, zero-extended) plus each channel of the
    send-bus mix (gains[n] * sends[n]) convolved with its IR, then the shared peak normalisation."""
    ir = np.atleast_2d(np.asarray(ir, dtype=np.float64))
    L = max(int(o) + len(w) for w, o in zip(waves, onsets))
    M = ir.shape[1]
    bus_gains = [float(g) * float(s) for g, s in zip(gains, sends)]
    if pans is None:
        dry = A.mix_arrangement(waves, onsets, gains, fades, track_len=L + M - 1)[None]
        bus = A.mix_arrangement(waves, onsets, bus_gains, fades, track_len=L)[None]
    else:
        dry = S.mix_stereo(waves, onsets, gains, pans, fades, track_len=L + M - 1)
        bus = S.mix_stereo(waves, onsets, bus_gains, pans, fades, track_len=L)
    out = dry + np.stack([fftconvolve(bus[c], ir[c if len(ir) == 2 else 0]) for c in range(len(bus))])
    if target_peak is not None:
        m = np.abs(out).max()
        if m > 0:
            out = out * (float(target_peak) / m)
    return out if pans is not None else out[0]


def render(waves_per_row, plan, ir, stereo: bool, target_peak=None) -> np.ndarray:
    """The chain after synthesis: every pitch item (row, semitones) of ``plan`` shifted by pitch_oracle.pitch_shift from its row's
    float64 waveform, then reverb_mix of the notes in plan order with the plan's per-note sends (and pans in stereo)."""
    shifted = [P.pitch_shift(waves_per_row[r], s) for r, s in plan.items]
    return reverb_mix([shifted[i] for i in plan.note_item], plan.onsets, plan.gains, plan.fades, plan.sends, ir,
                      plan.pans if stereo else None, target_peak)
