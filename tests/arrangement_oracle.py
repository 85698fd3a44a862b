"""CPU oracle of multi-instrument arrangements (TEST INFRASTRUCTURE ONLY): float64 numpy restatements of ds_mix_arrangement -- the
linear end-of-note fade, the ordered sum of every note of every track, and the peak normalisation -- on top of
tests/pitch_oracle.py, plus the expected TextToTimbre.arrangement_plan of a hand-written three-track case.

What is assumed (the reference's Track / DiffSynth mixing code is not available): tracks are summed plainly, a note fades out
linearly over its track's fade_out samples, and the piece is scaled so that its largest |sample| is the target peak."""
from __future__ import annotations

import numpy as np

from tests import pitch_oracle as P


def envelope(L: int, fade: int) -> np.ndarray:
    """Per-sample gain of a note of L samples with a fade of ``fade`` samples: 1 before the last F = min(fade, L) samples, then
    (L - i) / F, which is 1/F on the last sample; all ones for fade 0."""
    env = np.ones(L)
    F = min(int(fade), L)
    if F > 0:
        i = np.arange(L - F, L)
        env[L - F:] = (L - i) / F
    return env


def mix_arrangement(waves, onsets, gains, fades, target_peak=None, track_len=None) -> np.ndarray:
    """track[j] = sum over notes n in order of gains[n] * envelope_n(j - onsets[n]) * waves[n][j - onsets[n]], then, when target_peak
    is given and the track is not all zero, track * (target_peak / max |track|)."""
    n = max(int(o) + len(w) for w, o in zip(waves, onsets)) if track_len is None else int(track_len)
    track = np.zeros(n)
    for w, o, g, f in zip(waves, onsets, gains, fades):
        w = np.asarray(w, dtype=np.float64)
        track[int(o):int(o) + len(w)] += float(g) * envelope(len(w), f) * w
    if target_peak is not None:
        m = np.abs(track).max()
        if m > 0:
            track = track * (float(target_peak) / m)
    return track


def render(waves_per_row, plan, target_peak=None) -> np.ndarray:
    """The chain after synthesis: every pitch item (row, semitones) of ``plan`` shifted by pitch_oracle.pitch_shift from its row's
    float64 waveform, then mix_arrangement of the notes in plan order."""
    shifted = [P.pitch_shift(waves_per_row[r], s) for r, s in plan.items]
    return mix_arrangement([shifted[i] for i in plan.note_item], plan.onsets, plan.gains, plan.fades, target_peak)


# A hand-written arrangement: three tracks; durations 0.9 s (width 30) and 2.0 s (width 48) are used by two tracks each, 3.0 s
# (width 64) by one; (0.9 s, 0 semitones) repeats within track 0.  Latents and conditions are filled in by the caller.
HAND_NOTES = [
    ([(0.0, 0.9, 0, 1.0), (0.5, 2.0, -3, 0.5), (1.0, 0.9, 0, 0.5)], 0.5, 0.1),
    ([(0.25, 0.9, 7, 1.0), (1.5, 3.0, 12, 0.8)], 2.0, 0.0),
    ([(0.0, 2.0, 5, 0.25), (2.0, 2.0, 5, 1.0), (2.5, 2.0, -5, 1.0)], 1.0, 0.02),
]
HAND_PLAN = dict(
    rows=[(0, 0.9), (0, 2.0), (1, 0.9), (1, 3.0), (2, 2.0)],
    widths=[30, 48, 30, 64, 48],
    items=[(0, 0.0), (1, -3.0), (2, 7.0), (3, 12.0), (4, 5.0), (4, -5.0)],
    note_item=[0, 1, 0, 2, 3, 4, 4, 5],
    onsets=[0, 8000, 16000, 4000, 24000, 0, 32000, 40000],
    gains=[0.5, 0.25, 0.25, 2.0, 1.6, 0.25, 1.0, 1.0],
    fades=[1600, 1600, 1600, 0, 0, 320, 320, 320],
    lengths=[256 * 119, 256 * 191, 256 * 119, 256 * 119, 256 * 255, 256 * 191, 256 * 191, 256 * 191],
    track_len=24000 + 256 * 255,
)
