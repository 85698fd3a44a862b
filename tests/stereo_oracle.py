"""CPU oracle of stereo arrangements (TEST INFRASTRUCTURE ONLY): float64 numpy restatements of ds_mix_stereo -- the constant-power
pan law, the ordered two-channel sum of every note with its fade, and one peak normalisation for both channels -- on top of
tests/arrangement_oracle.py, plus the oracle chain after synthesis for a stereo TextToTimbre.arrangement_plan.

What is assumed (the reference has no stereo output): a note panned by p in [-1, 1] takes gains g cos(pi (1 + p) / 4) (left) and
g cos(pi (1 - p) / 4) (right), with cos(pi / 2) taken as exactly 0, and the piece is scaled by one factor so that its largest |sample|
over both channels is the target peak."""
from __future__ import annotations

import numpy as np

from tests import arrangement_oracle as A
from tests import pitch_oracle as P


def pan_cos(u: float) -> float:
    """cos(pi u / 4), with u == 2 (a hard pan to the other side) exactly 0: the float64 cos(pi / 2) is 6.1e-17."""
    return 0.0 if u == 2.0 else float(np.cos(np.pi * u / 4.0))


def pan_gains(gain: float, pan: float, fp32: bool = False):
    """(left, right) gains of a note of gain ``gain`` panned by ``pan``; ``fp32``: each rounded once to fp32, as the library does."""
    g, p = float(gain), float(pan)
    left, right = g * pan_cos(1.0 + p), g * pan_cos(1.0 - p)
    return (float(np.float32(left)), float(np.float32(right))) if fp32 else (left, right)


def mix_stereo(waves, onsets, gains, pans, fades, target_peak=None, track_len=None, fp32_gains: bool = False) -> np.ndarray:
    """[2, n]: channel c is arrangement_oracle.mix_arrangement of the notes with their channel-c pan gains; then, when target_peak is
    given and the piece is not all zero, both channels times target_peak / max |piece| over both."""
    lr = [pan_gains(g, p, fp32_gains) for g, p in zip(gains, pans)]
    out = np.stack([A.mix_arrangement(waves, onsets, [x[c] for x in lr], fades, track_len=track_len) for c in (0, 1)])
    if target_peak is not None:
        m = np.abs(out).max()
        if m > 0:
            out = out * (float(target_peak) / m)
    return out


def render(waves_per_row, plan, target_peak=None) -> np.ndarray:
    """The stereo chain after synthesis: every pitch item (row, semitones) of ``plan`` shifted by pitch_oracle.pitch_shift from its
    row's float64 waveform, then mix_stereo of the notes in plan order with the plan's per-note pans."""
    shifted = [P.pitch_shift(waves_per_row[r], s) for r, s in plan.items]
    return mix_stereo([shifted[i] for i in plan.note_item], plan.onsets, plan.gains, plan.pans, plan.fades, target_peak)
