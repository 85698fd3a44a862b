"""Spectral representation <-> waveform, batched on the GPU.

Replaces the per-sample CPU loop of the reference's decode glue
(webUI/natural_language_guided_4/utils.py:229-241: ``decode_stft`` -> ``depad_STFT`` -> ``librosa.istft``) and
encode glue (sound2sound_with_text.py:80-94: ``adjust_audio_length`` -> ``librosa.stft`` -> ``pad_STFT`` ->
``encode_stft``) with one fused kernel sequence each (ds_stft_decode_istft / ds_stft_encode), fp32."""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np
import torch

from . import _lib, ops
from ._lib import check


@torch.no_grad()
def spectrogram_to_waveform(spec: torch.Tensor) -> torch.Tensor:
    """[B,3,512,T] fp32 (log1p-magnitude, cos, sin) -> [B, 256*(T-1)] fp32."""
    spec = spec.float().contiguous()
    assert spec.dim() == 4 and spec.shape[1] == 3 and spec.shape[2] == 512, "expected [B,3,512,T]"
    B, T = spec.shape[0], spec.shape[3]
    lib = _lib.load()
    frames = torch.empty((B, T, 1024), dtype=torch.float32, device=spec.device)
    wave = torch.empty((B, lib.ds_istft_length(T)), dtype=torch.float32, device=spec.device)
    check(lib.ds_stft_decode_istft(spec.data_ptr(), frames.data_ptr(), wave.data_ptr(), B, T, ops._stream()), "ds_stft_decode_istft")
    return wave


def adjust_audio_length(audio, desired_length: int, original_sample_rate: Optional[int] = None, target_sample_rate: Optional[int] = None):
    """tools.adjust_audio_length (tools.py:126-151): resample when the rates differ, then crop or zero-pad the last axis.
    Tensors stay tensors, numpy arrays stay numpy arrays (drop-in use).  TextToTimbre.encode_audio resamples on the device instead
    (``resample_packed``, the Kaiser-sinc filter of ``resample``).
    The reference resamples with ``librosa.core.resample`` (absent from this image, un-pinned in requirements.txt:3; its default
    ``res_type`` is a band-limited sinc method): here a polyphase FIR resampler (``scipy.signal.resample_poly``) on the host
    -- parity of this branch is UNPINNED by necessity; it is one clip of host-side preprocessing, not part of the device path."""
    is_np = isinstance(audio, np.ndarray)
    if original_sample_rate is not None and target_sample_rate is not None and original_sample_rate != target_sample_rate:
        from math import gcd
        from scipy.signal import resample_poly
        g = gcd(int(original_sample_rate), int(target_sample_rate))
        a = audio if is_np else audio.detach().cpu().numpy()
        a = resample_poly(a, int(target_sample_rate) // g, int(original_sample_rate) // g, axis=-1)
        audio = a if is_np else torch.from_numpy(np.ascontiguousarray(a)).to(audio.device, audio.dtype)
    L = audio.shape[-1]
    if L >= desired_length:
        return audio[..., :desired_length]
    if is_np:
        out = np.zeros(audio.shape[:-1] + (desired_length,))          # the reference pads into np.zeros (float64), :146-148
        out[..., :L] = audio
        return out
    return torch.nn.functional.pad(audio, (0, desired_length - L))


# ---- numpy drop-ins of the reference's STFT+ helpers (tools.py:170-191, 320-345) ------------------------------------------------------
def pad_STFT(D: np.ndarray, time_resolution: Optional[int] = 256) -> np.ndarray:
    """tools.pad_STFT (:170-182): drop the DC row, zero-pad (never crop) the time axis to ``time_resolution``."""
    D = D[1:, :]
    if time_resolution is None:
        return D
    pad = time_resolution - D.shape[1]
    return np.pad(D, ((0, 0), (0, pad)), "constant") if pad > 0 else D


def depad_STFT(D_padded: np.ndarray) -> np.ndarray:
    """tools.depad_STFT (:185-191): prepend a zero DC row (float64 zeros, so complex64 input is promoted like the reference's)."""
    return np.concatenate([np.zeros((1, D_padded.shape[1])), D_padded], axis=0)


def _device():
    return torch.device("cuda", torch.cuda.current_device())


def _layout(x, item_dim: int, what: str = "unsupported layout"):
    """Host side of _pack: a list of ``item_dim``-D arrays / tensors (1-D signals, 2-D masks), one of them, or a batch of them
    along a leading axis -> (the arrays to pack, each item's shape, the layout for _unpack).  ValueError(``what``) for any other
    number of axes, and for an empty batch."""
    if isinstance(x, (list, tuple)):
        parts, kind = list(x), "list"
        shapes = [tuple(np.shape(a)) for a in parts]
        if any(len(s) != item_dim for s in shapes):
            raise ValueError(what)
    else:
        s = tuple(np.shape(x))
        if len(s) not in (item_dim, item_dim + 1):
            raise ValueError(what)
        parts, kind = [x], "one" if len(s) == item_dim else "batch"
        shapes = [s] if kind == "one" else [s[1:]] * s[0]
    if not shapes:
        raise ValueError("nothing to do: the batch is empty")
    return parts, shapes, (kind, isinstance(parts[0], np.ndarray))


def _pack(parts, device=None) -> torch.Tensor:
    """The arrays / tensors of _layout back to back in one fp32 tensor on ``device`` (by default the first one's CUDA device, else
    the current one)."""
    ts = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)) if isinstance(a, np.ndarray) else torch.as_tensor(a) for a in parts]
    dev = device if device is not None else ts[0].device if ts[0].is_cuda else _device()
    ts = [t.reshape(-1).to(dev, torch.float32) for t in ts]
    return torch.cat(ts) if len(ts) > 1 else ts[0]


def _unpack(out: torch.Tensor, shapes, layout):
    """A packed result whose items have ``shapes``, in the layout _layout read: a list, one item or a batch (numpy in, numpy out)."""
    kind, is_np = layout
    if kind == "list":
        parts = [p.view(s) for p, s in zip(torch.split(out, [int(np.prod(s)) for s in shapes]), shapes)]
        return [p.cpu().numpy() for p in parts] if is_np else parts
    res = out.view(shapes[0] if kind == "one" else (len(shapes),) + tuple(shapes[0]))
    return res.cpu().numpy() if is_np else res


def decode_stft(encoded_D: np.ndarray) -> np.ndarray:
    """tools.decode_stft (:334-345): [3, F, T] (log1p magnitude, cos, sin) -> complex [F, T], evaluated by ds_decode_stft in the
    precision of the input (float32 -> complex64, float64 -> complex128), like numpy."""
    enc = np.ascontiguousarray(encoded_D)
    dbl = enc.dtype == np.float64
    if not dbl:
        enc = enc.astype(np.float32, copy=False)
    t = torch.from_numpy(enc).to(_device())
    plane = int(np.prod(enc.shape[1:]))
    out = torch.empty(tuple(enc.shape[1:]) + (2,), dtype=t.dtype, device=t.device)
    check(_lib.load().ds_decode_stft(t.data_ptr(), out.data_ptr(), plane, 1 if dbl else 0, ops._stream()), "ds_decode_stft")
    return torch.view_as_complex(out).cpu().numpy()


def encode_stft(D: np.ndarray) -> np.ndarray:
    """tools.encode_stft (:320-331): complex [F, T] -> [3, F, T] (log1p|D|, cos angle, sin angle) by ds_encode_stft."""
    Dc = np.ascontiguousarray(D)
    dbl = Dc.dtype == np.complex128
    if not dbl:
        Dc = Dc.astype(np.complex64, copy=False)
    t = torch.view_as_real(torch.from_numpy(Dc)).contiguous().to(_device())
    plane = int(np.prod(Dc.shape))
    out = torch.empty((3,) + tuple(Dc.shape), dtype=t.dtype, device=t.device)
    check(_lib.load().ds_encode_stft(t.data_ptr(), out.data_ptr(), plane, 1 if dbl else 0, ops._stream()), "ds_encode_stft")
    return out.cpu().numpy()


def istft(D: np.ndarray, hop_length: int = 256, win_length: int = 1024) -> np.ndarray:
    """``librosa.istft(D, hop_length=256, win_length=1024)`` as the reference calls it (utils.py:184,241,260) for one complex
    [513, T] matrix (DC row ignored: depad_STFT made it zero), on the device through the fused decode + iSTFT kernel."""
    assert hop_length == 256 and win_length == 1024 and D.shape[0] == 513, "the path's iSTFT is fixed at n_fft 1024 / hop 256"
    enc = encode_stft(np.asarray(D)[1:].astype(np.complex64))
    return spectrogram_to_waveform(torch.from_numpy(enc)[None].to(_device()))[0].cpu().numpy()


@torch.no_grad()
def waveform_to_spectrogram(wave: torch.Tensor, time_resolution: int = 256) -> torch.Tensor:
    """[B, L] fp32 -> [B,3,512,time_resolution]: STFT(1024, hop 256, hann, centre zero-pad), DC row dropped,
    zero-padded in time, encoded as (log1p|D|, cos, sin)."""
    wave = wave.float().contiguous()
    B, L = wave.shape
    spec = torch.empty((B, 3, 512, time_resolution), dtype=torch.float32, device=wave.device)
    check(_lib.load().ds_stft_encode(wave.data_ptr(), L, spec.data_ptr(), B, time_resolution, ops._stream()), "ds_stft_encode")
    return spec


@torch.no_grad()
def griffinlim(magnitude: torch.Tensor, n_iter: int = 32, momentum: float = 0.99, init_phase: Optional[torch.Tensor] = None,
               generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """Magnitude-only reconstruction: ``librosa.griffinlim(abs_spec, n_iter=n_iter, hop_length=256, win_length=1024)`` as the
    reference's helpers call it (tools.py:63-76 ``save_results``, :194-217 ``nnData2Audio``, :220-223 ``amp_to_audio``;
    librosa defaults: momentum 0.99, random initial phases, centre zero padding), batched on the GPU from the fused STFT kernels.
    ``magnitude`` [B,512,T] holds bins 1..512 of the [513,T] matrix the reference builds (its DC row is zero, :205-210).
    ``init_phase`` [B,512,T] in radians replaces the random start (librosa draws it from an unseeded numpy generator)."""
    mag = magnitude.float().contiguous()
    assert mag.dim() == 3 and mag.shape[1] == 512, "expected [B,512,T]"
    B, _, T = mag.shape
    dev = mag.device
    if init_phase is None:
        init_phase = 2 * np.pi * torch.rand((B, 512, T), device=dev, generator=generator)
    ph = init_phase.to(dev, torch.float32)
    spec = torch.stack([torch.log1p(mag), torch.cos(ph), torch.sin(ph)], dim=1).contiguous()
    rebuilt = torch.empty_like(spec)
    tprev = torch.empty((B, 512, T, 2), dtype=torch.float32, device=dev)
    frames = torch.empty((B, T, 1024), dtype=torch.float32, device=dev)
    lib = _lib.load()
    L = lib.ds_istft_length(T)
    wave = torch.empty((B, L), dtype=torch.float32, device=dev)
    st = ops._stream()
    for it in range(n_iter):
        check(lib.ds_stft_decode_istft(spec.data_ptr(), frames.data_ptr(), wave.data_ptr(), B, T, st), "ds_stft_decode_istft")
        check(lib.ds_stft_encode(wave.data_ptr(), L, rebuilt.data_ptr(), B, T, st), "ds_stft_encode")
        check(lib.ds_griffinlim_update(rebuilt.data_ptr(), tprev.data_ptr(), spec.data_ptr(), float(momentum), 1 if it == 0 else 0, B, T, st),
              "ds_griffinlim_update")
    check(lib.ds_stft_decode_istft(spec.data_ptr(), frames.data_ptr(), wave.data_ptr(), B, T, st), "ds_stft_decode_istft")
    return wave


# ---- note arrangements: pitch shift and track mix (track_maker.py:42 and the placement loop after it) -------------------------
SAMPLE_RATE = 16000
MAX_SEMITONES = 24


def _check_steps(n_steps, count: int) -> np.ndarray:
    n = np.broadcast_to(np.asarray(n_steps, dtype=np.float64), (count,)).copy()
    if not np.all(np.isfinite(n)) or np.any(np.abs(n) > MAX_SEMITONES):
        raise ValueError(f"n_steps must be finite with |n_steps| <= {MAX_SEMITONES}, got {n_steps}")
    return n


@torch.no_grad()
def pitch_shift_packed(packed: torch.Tensor, lengths, n_steps, stages: Optional[dict] = None) -> torch.Tensor:
    """Batched pitch shift of items packed back to back in one fp32 device tensor (item k: lengths[k] samples) by n_steps[k]
    semitones (ds_pitch_shift); the result has the same layout.  ``stages`` (a dict, tests): receives the workspace and the byte
    offsets of the intermediate stages (see the header)."""
    lib = _lib.load()
    L = np.ascontiguousarray(lengths, dtype=np.int64)
    n = _check_steps(n_steps, len(L))
    packed = packed.float().contiguous()
    assert packed.dim() == 1 and packed.numel() == int(L.sum()), "packed length must equal the sum of the item lengths"
    nbytes, offs = C.c_longlong(0), (C.c_longlong * 4)()
    check(lib.ds_pitch_shift_workspace(L.ctypes.data, n.ctypes.data, len(L), C.byref(nbytes), offs), "ds_pitch_shift_workspace")
    ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=packed.device)
    out = torch.empty_like(packed)
    check(lib.ds_pitch_shift(packed.data_ptr(), out.data_ptr(), L.ctypes.data, n.ctypes.data, len(L), ws.data_ptr(), nbytes.value,
                             ops._stream()), "ds_pitch_shift")
    if stages is not None:
        stages.update(workspace=ws, offsets=list(offs))
    return out


def pitch_shift(waves, n_steps):
    """On-device, batched ``librosa.effects.pitch_shift(y, sr=16000, n_steps=n_steps, bins_per_octave=12)`` (track_maker.py:42)
    with librosa's default STFT arguments; the resampler is a Kaiser-windowed sinc (resampy kaiser_best) instead of librosa's soxr.
    ``waves``: a [B, L] or [L] tensor / numpy array, or a list of 1-D ones of different lengths; ``n_steps``: a scalar or one per
    item, finite, |n_steps| <= 24.  Returns the same layout (numpy in, numpy out; fp32)."""
    parts, shapes, layout = _layout(waves, 1, "expected [B, L], [L] or a list of 1-D signals")
    return _unpack(pitch_shift_packed(_pack(parts), [n for n, in shapes], n_steps), shapes, layout)


@torch.no_grad()
def mix_track(packed: torch.Tensor, src_offsets, lengths, onsets, gains, track_len: Optional[int] = None) -> torch.Tensor:
    """Place and sum notes into one fp32 track (ds_mix_track): note n is ``packed[src_offsets[n] : src_offsets[n] + lengths[n]]``
    times gains[n], starting at sample onsets[n]; notes may share a source.  Summed in note order, bit-identical run to run.
    ``track_len`` defaults to the end of the last note."""
    return _mix(packed, src_offsets, lengths, onsets, gains, track_len)


def _mix(packed: torch.Tensor, src_offsets, lengths, onsets, gains, track_len, fade: Optional[np.ndarray] = None,
         peak: float = 0.0, pans: Optional[np.ndarray] = None) -> torch.Tensor:
    """mix_track (``fade`` None: ds_mix_track), mix_arrangement (int64 ``fade``: ds_mix_arrangement, whose extra arguments are
    the fades before the note count and the peak after it) or mix_stereo (fp32 ``pans`` too: ds_mix_stereo, which takes the pans
    before the fades, and a [2, track_len] output): host arrays, workspace query, allocation, launch."""
    lib = _lib.load()
    off = np.ascontiguousarray(src_offsets, dtype=np.int64)
    L = np.ascontiguousarray(lengths, dtype=np.int64)
    on = np.ascontiguousarray(onsets, dtype=np.int64)
    g = np.ascontiguousarray(gains, dtype=np.float32)
    K = len(L)
    if track_len is None:
        track_len = int((on + L).max())
    if pans is not None:
        name, wk, fk = "ds_mix_stereo", (fade.ctypes.data, pans.ctypes.data, K, peak), (pans.ctypes.data, fade.ctypes.data, K, peak)
    else:
        name, fk = ("ds_mix_track", (K,)) if fade is None else ("ds_mix_arrangement", (fade.ctypes.data, K, peak))
        wk = fk
    nbytes = C.c_longlong(0)
    check(getattr(lib, name + "_workspace")(L.ctypes.data, on.ctypes.data, *wk, int(track_len), C.byref(nbytes)), name + "_workspace")
    packed = packed.float().contiguous()
    ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=packed.device)
    shape = (int(track_len),) if pans is None else (2, int(track_len))
    track = torch.empty(shape, dtype=torch.float32, device=packed.device)
    check(getattr(lib, name)(packed.data_ptr(), off.ctypes.data, L.ctypes.data, on.ctypes.data, g.ctypes.data, *fk, track.data_ptr(),
                             int(track_len), ws.data_ptr(), nbytes.value, ops._stream()), name)
    return track


def _check_peak(target_peak) -> float:
    """None (no normalisation) -> 0.0; otherwise a finite peak > 0."""
    if target_peak is None:
        return 0.0
    p = float(target_peak)
    if not np.isfinite(p) or p <= 0.0 or not np.isfinite(np.float32(p)):
        raise ValueError(f"target_peak must be None or a finite value > 0, got {target_peak}")
    return p


@torch.no_grad()
def mix_arrangement(packed: torch.Tensor, src_offsets, lengths, onsets, gains, fade_out, target_peak: Optional[float] = None,
                    track_len: Optional[int] = None) -> torch.Tensor:
    """mix_track with a linear fade over the last fade_out[n] samples of every note (clamped to the note; 0 = none) and, when
    ``target_peak`` is given, the track scaled on the device so that max |track| == target_peak (ds_mix_arrangement).  Notes
    without a fade are summed exactly as mix_track sums them.  Summed in note order, bit-identical run to run."""
    peak = _check_peak(target_peak)
    return _mix(packed, src_offsets, lengths, onsets, gains, track_len, _check_fades(fade_out), peak)


def _check_fades(fade_out) -> np.ndarray:
    """Per note: int64 samples >= 0."""
    fade = np.ascontiguousarray(fade_out, dtype=np.int64)
    if np.any(fade < 0):
        raise ValueError(f"fade_out must be >= 0, got {fade_out}")
    return fade


def _check_pans(pans, count: int) -> np.ndarray:
    """One fp32 pan per note, finite, in [-1, 1]."""
    p = np.ascontiguousarray(pans, dtype=np.float32).reshape(-1)
    if p.shape != (count,) or not np.all(np.isfinite(p)) or np.any(np.abs(p) > 1):
        raise ValueError(f"pans must be {count} finite values in [-1, 1], got {pans}")
    return p


@torch.no_grad()
def mix_stereo(packed: torch.Tensor, src_offsets, lengths, onsets, gains, pans, fade_out=None, target_peak: Optional[float] = None,
               track_len: Optional[int] = None) -> torch.Tensor:
    """mix_arrangement into two channels (ds_mix_stereo): note n is panned by pans[n] in [-1, 1] (-1 left, 0 centre, 1 right) with
    the constant-power law g_L = g cos(pi (1 + p) / 4), g_R = g cos(pi (1 - p) / 4), evaluated in float64 and rounded once, with a
    hard pan exactly 0 in the other channel.  ``fade_out``: None (no fades) or per note, as mix_arrangement takes it.  With
    ``target_peak``, both channels are scaled by one factor so that max |x| over both is the target.  Returns the planar fp32
    [2, track_len] (left, right); summed in note order, bit-identical run to run."""
    K = len(lengths)
    fade = np.zeros(K, dtype=np.int64) if fade_out is None else _check_fades(fade_out)
    return _mix(packed, src_offsets, lengths, onsets, gains, track_len, fade, _check_peak(target_peak), _check_pans(pans, K))


def shift_and_mix(sources, semitones, note_source, onsets, gains, fades=None, target_peak: Optional[float] = None,
                  pans=None, impulse_response: Optional[torch.Tensor] = None, sends=None) -> torch.Tensor:
    """The arrangement stage after synthesis: every source (1-D fp32 device tensor) is pitch-shifted by its semitones in ONE batched
    call, then note n -- source note_source[n] at sample onsets[n], scaled by gains[n] -- is mixed in ONE call.  Two library
    calls plus their workspace queries, whatever the number of notes.  ``pans`` (per note) mix through mix_stereo into [2, L];
    otherwise ``fades`` (per note, in samples) or ``target_peak`` mix through mix_arrangement; without either, through
    mix_track.

    ``impulse_response`` (an fp32 device tensor [H, M], H = 1, or 2 with ``pans``: left and right) adds convolution reverb: the
    result is dry + IR * bus, [L + M - 1] or [2, L + M - 1], where the dry mix is the mix above without its peak, zero past L, and
    the send bus is the same mix with gains[n] * sends[n] (post-fader, post-pan; ``sends`` per note, None = all 1).  One IR
    convolves every channel; two convolve left with left and right with right.  ``target_peak`` scales the sum, both channels by
    one factor.  Four library calls plus their workspace queries: the pitch shift, two mixes and one fftconvolve_packed."""
    lengths = [int(s.numel()) for s in sources]
    shifted = pitch_shift_packed(torch.cat([s.reshape(-1) for s in sources]), lengths, semitones)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    idx = np.asarray(note_source, dtype=np.int64)
    note_len = np.asarray(lengths, dtype=np.int64)[idx]
    if impulse_response is None:
        if pans is not None:
            return mix_stereo(shifted, starts[idx], note_len, onsets, gains, pans, fades, target_peak)
        if fades is None and target_peak is None:
            return mix_track(shifted, starts[idx], note_len, onsets, gains)
        fades = np.zeros(len(idx), dtype=np.int64) if fades is None else fades
        return mix_arrangement(shifted, starts[idx], note_len, onsets, gains, fades, target_peak)
    fades = np.zeros(len(idx), dtype=np.int64) if fades is None else fades
    L, (H, M) = int((np.asarray(onsets, dtype=np.int64) + note_len).max()), impulse_response.shape
    bus_gains = np.asarray(gains, dtype=np.float64) * (1.0 if sends is None else np.asarray(sends, dtype=np.float64))
    if pans is not None:
        dry = mix_stereo(shifted, starts[idx], note_len, onsets, gains, pans, fades, track_len=L + M - 1)
        bus = mix_stereo(shifted, starts[idx], note_len, onsets, bus_gains, pans, fades, track_len=L)
    else:
        dry = mix_arrangement(shifted, starts[idx], note_len, onsets, gains, fades, track_len=L + M - 1)
        bus = mix_arrangement(shifted, starts[idx], note_len, onsets, bus_gains, fades, track_len=L)
    ch = bus.numel() // L
    fftconvolve_packed(bus.reshape(-1), [L] * ch, impulse_response.reshape(-1), [M] * H, h_index=[0] * ch if H == 1 else [0, 1],
                       out=dry.reshape(-1), accumulate=True, target_peak=target_peak)
    return dry


# ---- convolution (scipy.signal.fftconvolve; reverb of arrangements) ------------------------------------------------------------
CONV_MODES = ("full", "same", "valid")


def fftconvolve_range(n: int, m: int, mode: str = "full"):
    """(start, length) of ``scipy.signal.fftconvolve(in1, in2, mode)`` for a 1-D in1 of n samples and in2 of m samples, within the
    full convolution of n + m - 1 samples: "full" (0, n + m - 1); "same", centred on in1, ((m - 1) // 2, n); "valid"
    (min(n, m) - 1, max(n, m) - min(n, m) + 1), which covers scipy's swap of the inputs when in2 is the longer."""
    if mode not in CONV_MODES:
        raise ValueError(f"mode must be one of {CONV_MODES}, got {mode!r}")
    n, m = int(n), int(m)
    if mode == "full":
        return 0, n + m - 1
    if mode == "same":
        return (m - 1) // 2, n
    return min(n, m) - 1, abs(n - m) + 1


@torch.no_grad()
def fftconvolve_packed(x: torch.Tensor, x_lengths, h: torch.Tensor, h_lengths, h_index=None, out_start=None, out_lengths=None,
                       out: Optional[torch.Tensor] = None, accumulate: bool = False, target_peak: Optional[float] = None) -> torch.Tensor:
    """Batched linear convolution by ds_fftconvolve: items packed back to back in the fp32 device tensor ``x`` (item k: x_lengths[k]
    samples), IRs packed in ``h`` (IR i: h_lengths[i] samples); item k is convolved with IR h_index[k] (default k) and writes
    out_lengths[k] samples of its full convolution starting at out_start[k] (default: the whole convolution), packed in item order.
    ``out``: an fp32 device tensor of that size to write into; ``accumulate`` adds the convolution to what ``out`` holds.
    ``target_peak`` scales every output of the call by one factor so that max |out| is the target."""
    lib = _lib.load()
    xl = np.ascontiguousarray(x_lengths, dtype=np.int64).reshape(-1)
    hl = np.ascontiguousarray(h_lengths, dtype=np.int64).reshape(-1)
    B, H = len(xl), len(hl)
    hi = np.arange(B, dtype=np.int64) if h_index is None else np.ascontiguousarray(np.broadcast_to(np.asarray(h_index, dtype=np.int64), (B,)))
    if ((hi < 0) | (hi >= H)).any():
        raise ValueError(f"h_index must be in [0, {H}), got {hi.tolist()}")
    st = np.zeros(B, dtype=np.int64) if out_start is None else np.ascontiguousarray(np.broadcast_to(np.asarray(out_start, dtype=np.int64), (B,)))
    ol = xl + hl[hi] - 1 - st if out_lengths is None else np.ascontiguousarray(np.broadcast_to(np.asarray(out_lengths, dtype=np.int64), (B,)))
    ol = np.ascontiguousarray(ol, dtype=np.int64)
    peak = _check_peak(target_peak)
    if accumulate and out is None:
        raise ValueError("accumulate=True needs an output tensor to add to")
    x = x.float().contiguous()
    h = h.to(x.device, torch.float32).contiguous()
    assert x.dim() == 1 and x.numel() == int(xl.sum()), "packed length of x must equal the sum of x_lengths"
    assert h.dim() == 1 and h.numel() == int(hl.sum()), "packed length of h must equal the sum of h_lengths"
    nbytes = C.c_longlong(0)
    check(lib.ds_fftconvolve_workspace(xl.ctypes.data, B, hl.ctypes.data, H, hi.ctypes.data, st.ctypes.data, ol.ctypes.data, peak,
                                       C.byref(nbytes)), "ds_fftconvolve_workspace")
    total = int(ol.sum())
    if out is None:
        out = torch.empty((total,), dtype=torch.float32, device=x.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == total and out.device == x.device
    ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=x.device)
    check(lib.ds_fftconvolve(x.data_ptr(), h.data_ptr(), out.data_ptr(), xl.ctypes.data, B, hl.ctypes.data, H, hi.ctypes.data,
                             st.ctypes.data, ol.ctypes.data, 1 if accumulate else 0, peak, ws.data_ptr(), nbytes.value, ops._stream()),
          "ds_fftconvolve")
    return out


def _check_impulse_response(ir, stereo: bool) -> torch.Tensor:
    """An impulse response as render_arrangement takes it -- [M], or with ``stereo`` [2, M] (left, right); a host or device tensor
    or a numpy array, finite and non-empty -> an fp32 CUDA tensor [H, M] (H = 1 or 2)."""
    t = torch.from_numpy(np.asarray(ir)) if isinstance(ir, np.ndarray) else torch.as_tensor(ir)
    if t.dim() == 2 and t.shape[0] == 2 and not stereo:
        raise ValueError("a [2, M] impulse response (left, right) needs stereo=True")
    if not (t.dim() == 1 or (t.dim() == 2 and t.shape[0] == 2)) or t.is_complex():
        raise ValueError(f"impulse_response must be a real [M] or, in stereo, [2, M] array, got shape {tuple(t.shape)}")
    if t.shape[-1] == 0:
        raise ValueError("impulse_response is empty")
    t = t.float().reshape(-1, t.shape[-1])
    if not bool(torch.isfinite(t).all()):
        raise ValueError("impulse_response must be finite in fp32")
    return t.to(t.device if t.is_cuda else _device()).contiguous()


def _check_sends(sends, count: int) -> np.ndarray:
    """One float64 reverb send level per track, finite and >= 0."""
    s = np.asarray(sends, dtype=np.float64).reshape(-1)
    if s.shape != (count,) or not np.all(np.isfinite(s)) or np.any(s < 0):
        raise ValueError(f"reverb_sends must be {count} finite values >= 0, got {sends}")
    return s


def _is_complex(a) -> bool:
    return a.is_complex() if torch.is_tensor(a) else np.iscomplexobj(a)


def _conv_operand(a, what: str):
    """The 1-D signals of one fftconvolve operand: a list of them, or an array / tensor of 1 or 2 axes (NotImplementedError for
    more batch axes and complex data, ValueError for an empty signal)."""
    is_list = isinstance(a, (list, tuple))
    items, max_nd = (list(a), 1) if is_list else ([a], 2)
    if any(np.ndim(t) > max_nd for t in items):
        raise NotImplementedError(f"{what}: only 1-D signals, or one batch axis before them, are implemented")
    if not items or any(np.ndim(t) < 1 for t in items):
        raise ValueError(f"{what}: expected 1-D signals, a [B, N] batch or a list of 1-D signals")
    if any(_is_complex(t) for t in items):
        raise NotImplementedError(f"{what}: complex inputs are not implemented")
    if any(0 in tuple(np.shape(t)) for t in items):
        raise ValueError(f"{what} is empty (scipy.signal.fftconvolve returns an empty array; this drop-in does not)")


def fftconvolve(in1, in2, mode: str = "full", axes=-1):
    """On-device, batched ``scipy.signal.fftconvolve(in1, in2, mode)`` along the last axis (ds_fftconvolve: partitioned FFTs in
    fp32).  ``in1``: [N], [B, N] or a list of 1-D signals; ``in2``: [M] or [1, M] (one IR for every item, transformed once),
    [B, M], or a list with one IR per item.  Modes are scipy's: "same" is centred on in1, "valid" has max(N, M) - min(N, M) + 1
    samples (fftconvolve_range).  The result has in1's layout (numpy in, numpy out; fp32).  Deviations: ``axes`` other than -1,
    complex data and more than one batch axis raise NotImplementedError, and an empty input raises ValueError where scipy returns
    an empty array."""
    if not (axes == -1 or (isinstance(axes, (list, tuple)) and list(axes) == [-1])):
        raise NotImplementedError(f"only axes=-1 is implemented, got {axes!r}")
    if mode not in CONV_MODES:
        raise ValueError(f"mode must be one of {CONV_MODES}, got {mode!r}")
    _conv_operand(in1, "in1")
    _conv_operand(in2, "in2")
    parts, shapes, layout = _layout(in1, 1, "expected [N], [B, N] or a list of 1-D signals")
    xl = [n for n, in shapes]
    B = len(xl)
    if isinstance(in2, (list, tuple)):
        hparts = list(in2)
    elif np.ndim(in2) == 1 or np.shape(in2)[0] == 1:
        hparts = [in2]
    else:
        hparts = [in2[i] for i in range(np.shape(in2)[0])]
    if len(hparts) not in (1, B):
        raise ValueError(f"in2 must hold one IR or one per item ({B}), got {len(hparts)}")
    hl = [int(np.shape(t)[-1]) for t in hparts]
    hi = [0] * B if len(hparts) == 1 else list(range(B))
    rng = [fftconvolve_range(n, hl[i], mode) for n, i in zip(xl, hi)]
    if layout[0] == "batch" and len({n for _, n in rng}) > 1:
        raise ValueError("a [B, N] input needs IRs that give every row the same output length; pass lists instead")
    x = _pack(parts)
    h = _pack([t.reshape(-1) if torch.is_tensor(t) else np.reshape(t, -1) for t in hparts], device=x.device)
    out = fftconvolve_packed(x, xl, h, hl, hi, [s for s, _ in rng], [n for _, n in rng])
    return _unpack(out, [(n,) for _, n in rng], layout)


# ---- sample-rate conversion (tools.adjust_audio_length's librosa.resample, tools.py:126-151) ----------------------------------
MAX_RATE = 4194304                      # DS_RESAMPLE_MAX_RATE


def _check_rates(sr, count: int, what: str) -> np.ndarray:
    """Integer sample rates, one per item (a scalar is broadcast); an integral float is accepted."""
    a = np.broadcast_to(np.asarray(sr, dtype=object), (count,))
    out = np.empty(count, dtype=np.int64)
    for k, v in enumerate(a):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)):
            raise ValueError(f"{what} must be an integer sample rate, got {v!r}")
        if not float(v).is_integer() or not 1 <= v <= MAX_RATE:
            raise ValueError(f"{what} must be an integer sample rate in 1..{MAX_RATE}, got {v!r}")
        out[k] = int(v)
    return out


def resample_length(length: int, orig_sr: int, target_sr: int) -> int:
    """librosa.resample's output length: ceil(length * (target_sr / orig_sr)) in float64 (not integer ceil-division)."""
    return int(np.ceil(length * (float(target_sr) / orig_sr)))


@torch.no_grad()
def resample_packed(packed: torch.Tensor, lengths, orig_sr, target_sr, out_lengths=None, normalize_peak: bool = False,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Batched resampling of items packed back to back in one fp32 device tensor (item k: lengths[k] samples, from orig_sr[k] to
    target_sr[k] Hz; rates: a scalar or one per item) by ds_resample.  Item k of the packed result has out_lengths[k] samples
    (librosa's length when None): zero-padded or cropped.  ``normalize_peak`` first divides each item by its peak |x|
    (at least 1e-12).  ``out``: an fp32 device tensor of the result's size to write into."""
    lib = _lib.load()
    L = np.ascontiguousarray(lengths, dtype=np.int64)
    B = len(L)
    o = _check_rates(orig_sr, B, "orig_sr")
    t = _check_rates(target_sr, B, "target_sr")
    ol = None if out_lengths is None else np.ascontiguousarray(np.broadcast_to(np.asarray(out_lengths, dtype=np.int64), (B,)))
    packed = packed.float().contiguous()
    assert packed.dim() == 1 and packed.numel() == int(L.sum()), "packed length must equal the sum of the item lengths"
    ol_ptr = None if ol is None else ol.ctypes.data
    nbytes = C.c_longlong(0)
    check(lib.ds_resample_workspace(L.ctypes.data, o.ctypes.data, t.ctypes.data, ol_ptr, B, C.byref(nbytes)), "ds_resample_workspace")
    total = int(ol.sum()) if ol is not None else sum(resample_length(n, a, b) for n, a, b in zip(L, o, t))
    if out is None:
        out = torch.empty((total,), dtype=torch.float32, device=packed.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == total and out.device == packed.device
    ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=packed.device)
    check(lib.ds_resample(packed.data_ptr(), out.data_ptr(), L.ctypes.data, o.ctypes.data, t.ctypes.data, ol_ptr,
                          1 if normalize_peak else 0, B, ws.data_ptr(), nbytes.value, ops._stream()), "ds_resample")
    return out


def resample(y, orig_sr, target_sr):
    """On-device, batched ``librosa.resample(y, orig_sr=orig_sr, target_sr=target_sr, res_type="kaiser_best")`` (resampy's
    Kaiser-windowed sinc, evaluated through a polyphase table; equal rates return the input).  ``y``: a [B, L] or [L] tensor /
    numpy array, or a list of 1-D ones of different lengths; rates: integers, a scalar or one per item.  The output has librosa's
    length ceil(L * target_sr / orig_sr) and the input's layout (numpy in, numpy out; fp32)."""
    parts, shapes, layout = _layout(y, 1, "expected [B, L], [L] or a list of 1-D signals")
    lengths = [n for n, in shapes]
    o, t = _check_rates(orig_sr, len(lengths), "orig_sr"), _check_rates(target_sr, len(lengths), "target_sr")
    n_out = [(resample_length(n, a, b),) for n, a, b in zip(lengths, o, t)]
    if layout[0] == "batch" and len(set(n_out)) > 1:
        raise ValueError("a [B, L] input needs rates that give every row the same output length; pass a list instead")
    return _unpack(resample_packed(_pack(parts), lengths, o, t), n_out, layout)


# ---- mask zoom (scipy.ndimage.zoom of the inpainting-with-text mask to the latent grid, inpaint_with_text.py) --------------------
MAX_ZOOM_DIM = 16384                    # DS_MASK_ZOOM_MAX_DIM


def _shapes(shapes, count: int, what: str) -> np.ndarray:
    """[count, 2] int64 from one (rows, cols) pair or one pair per item, every dimension in 1..MAX_ZOOM_DIM."""
    a = np.asarray(shapes, dtype=np.int64)
    if a.shape == (2,):
        a = np.broadcast_to(a, (count, 2))
    if a.shape != (count, 2):
        raise ValueError(f"{what} must be one (rows, cols) pair or one per item, got shape {a.shape}")
    if (a < 1).any() or (a > MAX_ZOOM_DIM).any():
        raise ValueError(f"every dimension of {what} must be in 1..{MAX_ZOOM_DIM}, got {a.tolist()}")
    return np.ascontiguousarray(a)


@torch.no_grad()
def zoom_packed(packed: torch.Tensor, in_shapes, out_shapes, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Batched ``scipy.ndimage.zoom`` (order 3, mode 'constant', prefilter, grid_mode False) of 2-D items packed back to back in
    one fp32 device tensor (item k: in_shapes[k] = (H, W), row-major) to out_shapes[k] = (h, w) (one pair, or one per item) by
    ds_mask_zoom, computed in float64 and rounded to fp32.  ``out``: a contiguous fp32 device tensor of the result's size to
    write into (any shape); the packed result otherwise."""
    lib = _lib.load()
    ins = np.asarray(in_shapes, dtype=np.int64).reshape(-1, 2)
    B = len(ins)
    ins = _shapes(ins, B, "in_shapes")
    outs = _shapes(out_shapes, B, "out_shapes")
    packed = packed.float().contiguous()
    assert packed.dim() == 1 and packed.numel() == int((ins[:, 0] * ins[:, 1]).sum()), "packed length must equal the sum of H * W"
    total = int((outs[:, 0] * outs[:, 1]).sum())
    if out is None:
        out = torch.empty((total,), dtype=torch.float32, device=packed.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == total and out.device == packed.device
    nbytes = C.c_longlong(0)
    check(lib.ds_mask_zoom_workspace(ins.ctypes.data, outs.ctypes.data, B, C.byref(nbytes)), "ds_mask_zoom_workspace")
    ws = torch.empty((nbytes.value,), dtype=torch.uint8, device=packed.device)
    check(lib.ds_mask_zoom(packed.data_ptr(), out.data_ptr(), ins.ctypes.data, outs.ctypes.data, B, ws.data_ptr(), nbytes.value,
                           ops._stream()), "ds_mask_zoom")
    return out


MORPH_PATHS = {"linear": 0, "slerp": 1}                # DS_MORPH_LINEAR, DS_MORPH_SLERP


@torch.no_grad()
def morph_rows(e0: torch.Tensor, e1: torch.Tensor, c0: torch.Tensor, c1: torch.Tensor, frames: int, path: str = "slerp"):
    """The initial-noise and condition rows of P timbre morphs of ``frames`` frames each, by one ds_morph_rows call: endpoints
    ``e0``, ``e1`` [P, n] and conditions ``c0``, ``c1`` [P, L] (fp32 device tensors of any shape whose leading axis is P) ->
    (noise [P*frames, n], conditions [P*frames, L]), row p*frames + k = frame k of sequence p at a = k / (frames - 1).
    ``path``: "linear" (the reference's generate_linear_noise, bit for bit) or "slerp" (spherical, conditions stay linear)."""
    if path not in MORPH_PATHS:
        raise ValueError(f"path must be one of {sorted(MORPH_PATHS)}, got {path!r}")
    lib = _lib.load()
    P = e0.shape[0]
    e0, e1 = e0.float().reshape(P, -1).contiguous(), e1.float().reshape(P, -1).contiguous()
    c0, c1 = c0.float().reshape(P, -1).contiguous(), c1.float().reshape(P, -1).contiguous()
    if e1.shape != e0.shape or c1.shape != c0.shape or c0.shape[0] != P:
        raise ValueError(f"endpoints must be [P, n] / [P, L] pairs of one P, got {tuple(e0.shape)}, {tuple(e1.shape)}, "
                         f"{tuple(c0.shape)}, {tuple(c1.shape)}")
    n, L, N, mode = e0.shape[1], c0.shape[1], int(frames), MORPH_PATHS[path]
    nbytes = C.c_longlong(0)
    check(lib.ds_morph_rows_workspace(P, N, n, L, mode, C.byref(nbytes)), "ds_morph_rows_workspace")
    noise = torch.empty((P * N, n), dtype=torch.float32, device=e0.device)
    cond = torch.empty((P * N, L), dtype=torch.float32, device=e0.device)
    ws = torch.empty((max(nbytes.value, 1),), dtype=torch.uint8, device=e0.device)
    check(lib.ds_morph_rows(e0.data_ptr(), e1.data_ptr(), c0.data_ptr(), c1.data_ptr(), P, N, n, L, mode, noise.data_ptr(),
                            cond.data_ptr(), ws.data_ptr(), nbytes.value, ops._stream()), "ds_morph_rows")
    return noise, cond


def zoom(input, zoom, output=None, order=3, mode="constant", cval=0.0, prefilter=True, *, grid_mode=False):
    """On-device, batched ``scipy.ndimage.zoom(input, zoom)`` for 2-D data with scipy's defaults; any other keyword value raises
    NotImplementedError.  ``input``: a [H, W] or [B, H, W] tensor / numpy array (B items of one shape), or a list of 2-D ones of
    different shapes; ``zoom``: a scalar or a (rows, cols) pair applied to every item, or for a list one per item.  Each item is
    ``round(H * zoom_rows) x round(W * zoom_cols)`` as in scipy, and the result has the input's layout (numpy in, numpy out; fp32)."""
    if output is not None or order != 3 or mode != "constant" or cval != 0.0 or prefilter is not True or grid_mode is not False:
        raise NotImplementedError("only scipy.ndimage.zoom's defaults (order=3, mode='constant', cval=0, prefilter=True, "
                                  "grid_mode=False, no output array) are implemented")
    parts, ins, layout = _layout(input, 2, "expected a [H, W] or [B, H, W] array, or a list of 2-D arrays")
    B, is_list = len(ins), layout[0] == "list"
    z = np.asarray(zoom, dtype=np.float64)
    if z.ndim == 0:
        z = np.full((B, 2), float(z))
    elif z.shape == (2,):
        z = np.broadcast_to(z, (B, 2))
    elif is_list and z.shape == (B,):
        z = np.repeat(z[:, None], 2, axis=1)
    elif not (is_list and z.shape == (B, 2)):
        raise ValueError(f"zoom must be a scalar or a (rows, cols) pair{', or one per item' if is_list else ''}, got {zoom!r}")
    if not np.all(np.isfinite(z)) or (z <= 0).any():
        raise ValueError(f"zoom factors must be finite and positive, got {zoom!r}")
    outs = [tuple(int(round(n * f)) for n, f in zip(s, zk)) for s, zk in zip(ins, z)]        # scipy: round(n * zoom), Python's round
    in_shapes, out_shapes = _shapes(ins, B, "the input shape"), _shapes(outs, B, "the output shape")
    return _unpack(zoom_packed(_pack(parts), in_shapes, out_shapes), outs, layout)


@torch.no_grad()
def spectrogram_images(spec: torch.Tensor):
    """[B,3,512,T] fp32 spectral representation -> (dB-magnitude image, phase image), uint8 [B,513,T,3] each: what
    ``spectrogram_to_Gradio_image(np.abs(D))`` / ``phase_to_Gradio_image(np.angle(D))`` (utils.py:8-91) give for
    ``D = depad_STFT(decode_stft(spec[b]))`` (utils.py:229-238), for the whole batch in two kernels."""
    spec = spec.float().contiguous()
    assert spec.dim() == 4 and spec.shape[1] == 3 and spec.shape[2] == 512, "expected [B,3,512,T]"
    B, T = spec.shape[0], spec.shape[3]
    mag = torch.empty((B, 513, T, 3), dtype=torch.uint8, device=spec.device)
    ph = torch.empty_like(mag)
    scratch = torch.empty((B,), dtype=torch.int64, device=spec.device)
    check(_lib.load().ds_spec_images(spec.data_ptr(), mag.data_ptr(), ph.data_ptr(), scratch.data_ptr(), B, T, ops._stream()),
          "ds_spec_images")
    return mag, ph


@torch.no_grad()
def latent_images(latents: torch.Tensor) -> torch.Tensor:
    """[B,4,H,W] fp32 -> uint8 [B,8H,8W,4] (latent_representation_to_Gradio_image, utils.py:94-128, batched;
    the input is left untouched -- the reference normalises its numpy argument in place)."""
    lat = latents.float().contiguous()
    assert lat.dim() == 4 and lat.shape[1] == 4, "expected [B,4,H,W]"
    B, _, H, W = lat.shape
    img = torch.empty((B, 8 * H, 8 * W, 4), dtype=torch.uint8, device=lat.device)
    scratch = torch.empty((B, 4, 2), dtype=torch.float32, device=lat.device)
    check(_lib.load().ds_latent_image(lat.data_ptr(), img.data_ptr(), scratch.data_ptr(), B, H, W, ops._stream()), "ds_latent_image")
    return img


def latent_representation_to_Gradio_image(latent_representation) -> np.ndarray:
    """Drop-in for utils.py:94-128: one latent [4,H,W] (tensor or numpy) -> uint8 [8H,8W,4] numpy."""
    if isinstance(latent_representation, np.ndarray):
        latent_representation = torch.from_numpy(latent_representation)
    dev = latent_representation.device if latent_representation.is_cuda else torch.device("cuda", torch.cuda.current_device())
    return latent_images(latent_representation.to(dev)[None])[0].cpu().numpy()


def _decode_lists(spec: torch.Tensor):
    mag, ph = spectrogram_images(spec)
    wave = spectrogram_to_waveform(spec)
    mag, ph, wave = mag.cpu().numpy(), ph.cpu().numpy(), wave.cpu().numpy()
    return [m for m in mag], [p for p in ph], [w for w in wave]


@torch.no_grad()
def encodeBatch2GradioOutput_STFT(decoder, latent_vector_batch, resolution=(512, 256), original_STFT_batch=None):
    """utils.py:194-267 without the per-sample CPU loop.  Returns the reference's 6 lists
    (dB-spectrogram images, phase images, signals, and the same three with channel 0 of the reconstruction replaced by
    ``original_STFT_batch``'s when that is given, else empty).  Images are uint8 [513,T,3] numpy arrays; signals are
    float32 numpy arrays (the reference's are float64)."""
    if isinstance(latent_vector_batch, np.ndarray):
        latent_vector_batch = torch.from_numpy(latent_vector_batch).to(next(decoder.parameters()).device)
    rec = decoder(latent_vector_batch)
    imgs, phases, signals = _decode_lists(rec)
    if original_STFT_batch is None:
        return imgs, phases, signals, [], [], []
    if isinstance(original_STFT_batch, np.ndarray):
        original_STFT_batch = torch.from_numpy(original_STFT_batch)
    swapped = rec.float().clone()
    swapped[:, 0] = original_STFT_batch[:, 0].to(rec.device, torch.float32)          # utils.py:251
    return (imgs, phases, signals) + _decode_lists(swapped)


@torch.no_grad()
def InputBatch2Encode_STFT(encoder, STFT_batch, resolution=(512, 256), quantizer=None, squared=True):
    """utils.py:131-191: encode a batch of spectral representations (and quantise), and render the INPUT batch back to
    images / signals.  ``quantizer=None`` is the reference's VAE branch (:162-164): the encoder must then return
    ``(mu, logvar, z)`` and there is no quantised batch; the deployed VQGAN encoder returns a single tensor, so -- exactly as
    in the reference -- that combination fails at the unpacking."""
    device = next(encoder.parameters()).device
    if isinstance(STFT_batch, np.ndarray):
        STFT_batch = torch.from_numpy(STFT_batch)
    spec = STFT_batch.to(device, torch.float32)
    if quantizer is not None:
        latents = encoder(spec)
        quantized, _loss, (_, _, _) = quantizer(latents)
    else:
        _mu, _logvar, latents = encoder(spec)          # (a tensor [3, ...] would be split along dim 0, as in the reference)
        quantized = None
    imgs, phases, signals = _decode_lists(spec)
    return imgs, phases, signals, latents, quantized
