"""CPU oracle of the note-arrangement path (TEST INFRASTRUCTURE ONLY): float64 numpy restatements of what track_maker.DiffSynth does
after its per-note closure -- ``librosa.effects.pitch_shift`` per note (track_maker.py:42), then gain, placement and sum.

Third-party arithmetic (librosa, absent here).  librosa.effects.pitch_shift(y, sr=16000, n_steps=n, bins_per_octave=12) with
librosa's default STFT arguments (n_fft 2048, hop 512, periodic Hann, centre zero padding) is restated exactly except for the
resampler: librosa's default is soxr, which cannot be restated; ``resample_kaiser`` is the Kaiser-windowed sinc of resampy's
kaiser_best (librosa's default before 0.10), so parity with librosa is unpinned, as for Griffin-Lim.  The STFT is
``oracle.ds_oracle.stft``; the iSTFT with librosa's ``length`` semantics (``istft_length``) is pinned against ``torch.istft`` in
float64 (tests/test_track_oracle.py)."""
from __future__ import annotations

import numpy as np

from oracle.ds_oracle import hann_periodic, stft

SR = 16000
RS_ZEROS, RS_ROLLOFF, RS_BETA = 64, 0.9475937167399596, 14.769656459379492


def fix_length(y: np.ndarray, size: int) -> np.ndarray:
    """librosa.util.fix_length on the last axis: trim or zero-pad to ``size``."""
    if y.shape[-1] >= size:
        return y[..., :size]
    return np.concatenate([y, np.zeros(y.shape[:-1] + (size - y.shape[-1],))], axis=-1)


def istft_length(D: np.ndarray, hop: int, length: int) -> np.ndarray:
    """librosa.istft(D, hop_length=hop, length=length) (center=True, window='hann'): n_fft = 2*(rows-1); only the first
    ceil((length + n_fft)/hop) frames are used; per-frame irfft * window; overlap-add; divide by the overlap-added squared window
    where it exceeds ``tiny``; drop n_fft//2 samples at the start; zero-pad or trim to ``length``."""
    n_fft = 2 * (D.shape[0] - 1)
    D = D[:, :min(D.shape[1], int(np.ceil((length + 2 * (n_fft // 2)) / hop)))]
    T = D.shape[1]
    w = hann_periodic(n_fft)
    frames = np.fft.irfft(D.astype(np.complex128), n=n_fft, axis=0) * w[:, None]
    total = n_fft + hop * (T - 1)
    y = np.zeros(total)
    wss = np.zeros(total)
    for t in range(T):
        y[t * hop:t * hop + n_fft] += frames[:, t]
        wss[t * hop:t * hop + n_fft] += w * w
    ok = wss > np.finfo(np.float64).tiny
    y[ok] /= wss[ok]
    return fix_length(y[n_fft // 2:], length)


def phase_vocoder(D: np.ndarray, rate: float, hop: int = 512) -> np.ndarray:
    """librosa.phase_vocoder(D, rate=rate, hop_length=hop) for one complex [bins, T] matrix."""
    time_steps = np.arange(0, D.shape[-1], rate, dtype=np.float64)
    out = np.zeros((D.shape[0], len(time_steps)), dtype=np.complex128)
    phi_advance = np.linspace(0, np.pi * hop, D.shape[0])
    phase_acc = np.angle(D[:, 0])
    Dp = np.pad(D, [(0, 0), (0, 2)], mode="constant")
    for t, step in enumerate(time_steps):
        columns = Dp[:, int(step):int(step + 2)]
        alpha = np.mod(step, 1.0)
        mag = (1.0 - alpha) * np.abs(columns[:, 0]) + alpha * np.abs(columns[:, 1])
        out[:, t] = mag * np.exp(1.0j * phase_acc)
        dphase = np.angle(columns[:, 1]) - np.angle(columns[:, 0]) - phi_advance
        dphase = dphase - 2.0 * np.pi * np.round(dphase / (2.0 * np.pi))
        phase_acc = phase_acc + phi_advance + dphase
    return out


def time_stretch(y: np.ndarray, rate: float) -> np.ndarray:
    """librosa.effects.time_stretch(y, rate=rate): stft(2048, 512) -> phase_vocoder -> istft(length=round(len(y)/rate))."""
    D = stft(y, n_fft=2048, hop=512)
    return istft_length(phase_vocoder(D, rate, hop=512), hop=512, length=int(round(len(y) / rate)))


def resample_kaiser(y: np.ndarray, ratio: float, zeros: int = RS_ZEROS, rolloff: float = RS_ROLLOFF, beta: float = RS_BETA) -> np.ndarray:
    """Band-limited resampling by ``ratio`` (target rate / source rate) with the filter of resampy's kaiser_best, evaluated directly
    (no table): out[j] = sum_i y[i] h(i - j/ratio), h(d) = s*rolloff*sinc(s*rolloff*d) * I0(beta*sqrt(1-(s*d/zeros)^2)) / I0(beta)
    for |d| <= zeros/s, s = min(1, ratio); samples outside [0, len) count as zero; ceil(len*ratio) outputs.  Vectorised over the
    output samples, one pass per tap offset."""
    from scipy.special import i0
    y = np.asarray(y, dtype=np.float64)
    n_out = int(np.ceil(len(y) * ratio))
    sc = min(1.0, ratio)
    half, cut = zeros / sc, rolloff * sc
    pos = np.arange(n_out) / ratio
    ip = np.floor(pos)
    f = pos - ip
    ip = ip.astype(np.int64)
    out = np.zeros(n_out)
    inv_i0 = 1.0 / i0(beta)
    M = int(np.ceil(half)) + 1
    for m in range(-M, M + 1):
        d = m - f
        i = ip + m
        ok = (np.abs(d) <= half) & (i >= 0) & (i < len(y))
        if not ok.any():
            continue
        dk = d[ok]
        u = dk * (sc / zeros)
        h = cut * np.sinc(cut * dk) * i0(beta * np.sqrt(np.clip(1.0 - u * u, 0.0, None))) * inv_i0
        out[ok] += y[i[ok]] * h
    return out


def pitch_shift(y: np.ndarray, n_steps: float, sr: int = SR) -> np.ndarray:
    """librosa.effects.pitch_shift(y, sr=sr, n_steps=n_steps, bins_per_octave=12) with resample_kaiser in place of soxr:
    time_stretch by rate = 2^(-n_steps/12), resample from sr/rate to sr (skipped when the rates are equal), fix_length(len(y))."""
    assert np.isfinite(n_steps) and abs(n_steps) <= 24
    y = np.asarray(y, dtype=np.float64)
    rate = 2.0 ** (-float(n_steps) / 12.0)
    ys = time_stretch(y, rate)
    if rate != 1.0:
        ys = resample_kaiser(ys, rate)
    return fix_length(ys, len(y))


def mix_track(waves, onsets, gains) -> np.ndarray:
    """The placement loop: track[j] = sum_k gains[k] * waves[k][j - onsets[k]] (onsets in samples), summed in note order; the
    track ends with the last note; no normalisation, no envelope."""
    n = max(int(o) + len(w) for w, o in zip(waves, onsets))
    track = np.zeros(n)
    for w, o, g in zip(waves, onsets, gains):
        track[int(o):int(o) + len(w)] += float(g) * np.asarray(w, dtype=np.float64)
    return track
