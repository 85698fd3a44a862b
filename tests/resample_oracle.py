"""CPU oracle of sample-rate conversion (TEST INFRASTRUCTURE ONLY): float64 numpy restatements of
``librosa.resample(y, orig_sr, target_sr, res_type="kaiser_best")`` as the timbre-modification upload handler calls it through
tools.adjust_audio_length (tools.py:126-151, sound2sound_with_text.py:75-82).

Third-party arithmetic (librosa, absent here).  ``resample`` uses ``tests.pitch_oracle.resample_kaiser``, the Kaiser-windowed sinc of
resampy's kaiser_best evaluated directly (not librosa's default soxr, so parity with librosa is unpinned, as for the pitch shift),
with librosa's float64 output length and the input itself at equal rates; ``resample_polyphase`` restates it with the phases
indexed in integers as the device does; ``upload_chain`` is normalise -> resample -> fix_length -> ``oracle.ds_oracle``'s STFT
encode.  Pinned against analytic resampling of band-limited tones in tests/test_resample_oracle.py."""
from __future__ import annotations

import numpy as np

from tests.pitch_oracle import RS_BETA, RS_ROLLOFF, RS_ZEROS, SR, fix_length, resample_kaiser

__all__ = ["RS_BETA", "RS_ROLLOFF", "RS_ZEROS", "SR", "fix_length", "resample_kaiser", "resample_length", "resample", "polyphase_table",
           "resample_polyphase", "upload_chain"]


def resample_length(n: int, orig_sr: int, target_sr: int) -> int:
    """librosa.resample's output length: int(np.ceil(n * float(target_sr) / orig_sr)), float64."""
    return int(np.ceil(n * (float(target_sr) / orig_sr)))


def resample(y: np.ndarray, orig_sr: int, target_sr: int) -> np.ndarray:
    """librosa.resample(y, orig_sr=orig_sr, target_sr=target_sr, res_type="kaiser_best") with resampy's filter evaluated directly
    (``resample_kaiser``): librosa's output length, and the input itself when the rates are equal."""
    y = np.asarray(y, dtype=np.float64)
    if orig_sr == target_sr:
        return y.copy()
    out = resample_kaiser(y, float(target_sr) / orig_sr)
    assert len(out) == resample_length(len(y), orig_sr, target_sr)
    return out


def polyphase_table(orig_sr: int, target_sr: int, zeros: int = RS_ZEROS, rolloff: float = RS_ROLLOFF, beta: float = RS_BETA):
    """The coefficient table of the integer-rate resampler: with g = gcd, up = target/g, down = orig/g and F = floor(zeros/s),
    row p (phase p/up) holds h(m - p/up) for m = -F .. F+1 (zero outside the filter's support).  Returns (table, up, down, F)."""
    from math import gcd
    from scipy.special import i0
    g = gcd(orig_sr, target_sr)
    up, down = target_sr // g, orig_sr // g
    sc = min(1.0, float(target_sr) / orig_sr)
    half, cut = zeros / sc, rolloff * sc
    F = int(np.floor(half))
    m = np.arange(-F, F + 2, dtype=np.float64)
    d = m[None, :] - (np.arange(up, dtype=np.float64) / up)[:, None]
    u = d * (sc / zeros)
    h = cut * np.sinc(cut * d) * i0(beta * np.sqrt(np.clip(1.0 - u * u, 0.0, None))) / i0(beta)
    # support |m - p/up| <= zeros/s decided in integers, |m*up - p| <= zeros*max(up, down): the ties at the edge are exact
    reach = np.abs(np.arange(-F, F + 2, dtype=np.int64)[None, :] * up - np.arange(up, dtype=np.int64)[:, None])
    return np.where(reach <= zeros * max(up, down), h, 0.0), up, down, F


def resample_polyphase(y: np.ndarray, orig_sr: int, target_sr: int) -> np.ndarray:
    """``resample`` restated as the device computes it: output j has base input (j*down) div up and phase (j*down) mod up, both in
    integer arithmetic, and sums y[base + m] * table[phase][m + F] over m = -F .. F+1 in ascending order."""
    y = np.asarray(y, dtype=np.float64)
    if orig_sr == target_sr:
        return y.copy()
    tab, up, down, F = polyphase_table(orig_sr, target_sr)
    n_out = resample_length(len(y), orig_sr, target_sr)
    jd = np.arange(n_out, dtype=np.int64) * down
    base, phase = jd // up, jd % up
    yp = np.concatenate([np.zeros(F), y, np.zeros(F + 2 + int(base[-1]) + 1)])       # y[i] at yp[i + F]; zeros outside
    out = np.zeros(n_out)
    for c in range(2 * F + 2):                                                          # tap m = c - F
        out += yp[base + c] * tab[phase, c]
    return out


def upload_chain(y: np.ndarray, orig_sr: int, width: int = 64):
    """The upload handler's chain (sound2sound_with_text.py:75-94) with ``resample``: peak-normalise (peak at least 1e-12),
    resample to 16 kHz, fix_length to 256*(4w-1), then ds_oracle's stft -> pad_STFT -> encode_stft at max(256, 4w) frames.
    Returns (encoder input waveform, [3, 512, T] spectrogram)."""
    from oracle.ds_oracle import waveform_to_spectrogram
    y = np.asarray(y, dtype=np.float64)
    y = y / max(np.abs(y).max(), 1e-12)
    wave = fix_length(resample(y, orig_sr, SR), 256 * (4 * width - 1))
    return wave, waveform_to_spectrogram(wave, time_resolution=max(256, 4 * width))
