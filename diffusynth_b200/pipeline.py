"""Text-to-timbre pipeline (the hot path of webUI/natural_language_guided_4/text2sound.py:45-179, without the UI):
condition vectors -> DiffSynthSampler.sample (CFG, respaced DDIM/DDPM) -> VectorQuantizerEMA -> Decoder ->
STFT+ decode + iSTFT -> waveforms, and its data-parallel form (prompts sharded over ranks, one all-gather)."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib, ops, weights as W
from ._lib import check
from .codec import MORPH_PATHS, SAMPLE_RATE, _check_impulse_response, _check_peak, _check_sends, _layout, _pack, morph_rows, resample_packed, shift_and_mix, \
    spectrogram_to_waveform, waveform_to_spectrogram, zoom_packed
from .sampler import DiffSynthSampler
from .unet import ConditionedUnet
from .vqgan import VQGAN


@dataclass
class Timbres:
    latents: torch.Tensor        # [B,4,128,W]     final continuous latent (imgs[-1])
    quantized: torch.Tensor      # [B,4,128,W]
    spectrograms: torch.Tensor   # [B,3,512,4W]
    waveforms: torch.Tensor      # [B, 256*(4W-1)]
    initial_noise: Optional[torch.Tensor] = None     # [B,4,128,64] train-width noise each row started from


@dataclass
class TrackPlan:
    durations: list              # distinct note durations (s), in order of first appearance
    pairs: list                  # distinct (index into durations, semitones), in order of first appearance
    note_pair: list              # per note: index into pairs
    onsets: list                 # per note: onset in samples
    gains: list                  # per note
    lengths: list                # per note: samples of its waveform, 256 * (4 * width - 1)
    track_len: int               # max(onset + length)


@dataclass
class ArrangementPlan:
    rows: list                   # distinct (track, duration (s)): tracks in order, durations in order of first appearance
    widths: list                 # per row: latent width
    items: list                  # distinct (index into rows, semitones), in order of first appearance
    note_item: list              # per note (tracks in order, then notes in order): index into items
    onsets: list                 # per note: onset in samples
    gains: list                  # per note: note gain * track gain
    fades: list                  # per note: fade-out of its track in samples
    lengths: list                # per note: samples of its waveform, 256 * (4 * width - 1)
    track_len: int               # max(onset + length) over every track
    pans: list = field(default_factory=list)   # per note: pan of its track, in [-1, 1] (0 for a 5-tuple track)
    sends: list = field(default_factory=list)  # per note: reverb send level of its track (1.0 without reverb_sends)


class _Tail:
    """quantiser -> decoder -> STFT+ decode + iSTFT (text2sound.py:128-134, utils.py:224-241) as a fixed launch sequence on
    static buffers, so that it is captured in the same CUDA graph as the sampling loop: ``src`` is the loop's final-latent
    buffer; the quantiser writes straight into the decoder plan's input, the iSTFT reads the decoder plan's output."""

    def __init__(self, vqgan: VQGAN, src: torch.Tensor):
        B, Cc, H, Wd = src.shape
        dev = src.device
        lib = _lib.load()
        self.src = src
        self.dec = vqgan._decoder._stack.plan(B, H, Wd)
        self.q = self.dec.inp                                   # [B,4,H,W] fp32: decoder input = quantiser output
        self.idx = torch.empty((B * H * Wd,), dtype=torch.long, device=dev)
        self.spec = self.dec.out_f32                            # [B,3,4H,4W]
        T = self.spec.shape[3]
        self.frames = torch.empty((B, T, 1024), dtype=torch.float32, device=dev)
        self.wave = torch.empty((B, lib.ds_istft_length(T)), dtype=torch.float32, device=dev)
        vq = vqgan._vq_vae
        K = vq._num_embeddings
        self.ops = [("vq", lambda: vq.quantize_into(self.src, self.q, self.idx))] + list(self.dec.ops) + [
            ("istft", lambda: check(lib.ds_stft_decode_istft(self.spec.data_ptr(), self.frames.data_ptr(), self.wave.data_ptr(), B, T,
                                                             ops._stream()), "ds_stft_decode_istft"))]
        self.meta = dict(self.dec.meta)
        # the quantiser is fp32-ALU work: 4 FMAs per (position, code) for the dot product + the compare (VQGAN.py:107-112)
        self.meta["vq"] = dict(family="vq_quantize", flops=0.0, bytes=B * H * Wd * (2 * Cc * 4.0 + 8.0), fp32_flops=B * H * Wd * K * 2.0 * Cc)
        self.meta["istft"] = dict(family="istft(decode+frames+ola)", flops=0.0, bytes=B * (3 * 512 * T * 4.0 + self.wave.shape[1] * 4.0))
        self.num_launches = len(self.ops) + 1 + sum(1 for n, _ in self.ops if n.endswith(".fin"))      # iSTFT = 2 kernels, finalize = 2

    def run(self):
        for _, fn in self.ops:
            fn()


class _TailBuffers:
    """Result buffers of the tail when it runs inside the library's sampling graph (ds_sample_graph_build): the same attributes
    _Tail exposes (q, idx, spec, wave), no launch list."""

    def __init__(self, src: torch.Tensor):
        B, Cc, H, Wd = src.shape
        dev = src.device
        self.src = src
        self.q = torch.empty((B, Cc, H, Wd), dtype=torch.float32, device=dev)
        self.idx = torch.empty((B * H * Wd,), dtype=torch.long, device=dev)
        self.spec = torch.empty((B, 3, 4 * H, 4 * Wd), dtype=torch.float32, device=dev)
        self.wave = torch.empty((B, _lib.load().ds_istft_length(4 * Wd)), dtype=torch.float32, device=dev)


class _TailFactory:
    """What the sampler needs to put the tail into its graph: the VQGAN (its module-level handle for the library's graph), the
    result buffers, or -- for the operator-level path and bench.py's per-kernel timings -- the Python launch list."""

    def __init__(self, vqgan: VQGAN):
        self.vqgan = vqgan

    def __call__(self, src: torch.Tensor) -> _Tail:
        return _Tail(self.vqgan, src)

    def buffers(self, src: torch.Tensor) -> _TailBuffers:
        return _TailBuffers(src)


class TextToTimbre:
    def __init__(self, unet: ConditionedUnet, vqgan: VQGAN, timesteps: int = 1000, height: int = 128, channels: int = 4,
                 noise_strategy: str = "repeat", device=None):
        self.unet, self.vqgan = unet, vqgan
        self.timesteps, self.height, self.channels, self.noise_strategy = timesteps, height, channels, noise_strategy
        self.device = torch.device(device if device is not None else unet.device)
        self._samplers = {}
        self._tail_factory = _TailFactory(self.vqgan)                # one object: its id() is part of the samplers' graph keys
        self.last_launches = 0
        self._last_tail: Optional[_Tail] = None

    def tail_for(self, batch: int, width: int) -> _Tail:
        """The tail of the most recent generate() of this batch / width as an operator-level launch list on the same final-latent
        buffer (bench.py times its launches one by one)."""
        t = self._last_tail
        assert t is not None and t.src.shape[0] == batch and t.src.shape[3] == width, "no generate() call with this shape yet"
        return t if isinstance(t, _Tail) else _Tail(self.vqgan, t.src)

    def _run(self, s: DiffSynthSampler, call, B: int, noise_feed, decode: bool) -> Timbres:
        """One sampling call of B rows on ``s`` (guidance already active): ``call(initial_noise)`` runs the sampler's entry point;
        ``noise_feed`` as generate takes it.  With ``decode`` the quantiser (text2sound.py:128), decoder (utils.py:224) and iSTFT
        (utils.py:229-241) run in the sampling graph and their results are copied out of its static buffers."""
        init = None
        s.noise_feed = None
        if noise_feed is not None:
            init = noise_feed[0][:B].to(self.device, torch.float32)
            s.noise_feed = noise_feed[1:] if len(noise_feed) > 1 else None
        s.graph_tail, s.final_only = (self._tail_factory if decode else None), True
        imgs, _ = call(init)
        self.last_launches = s.last_graph_launches
        if not decode:
            return Timbres(imgs[-1], None, None, None, s.last_reference_noise)
        t = s.last_tail
        self._last_tail = t
        self.vqgan._vq_vae.last_indices = t.idx.clone()
        return Timbres(imgs[-1], t.q.clone(), t.spec.clone(), t.wave.clone(), s.last_reference_noise)

    def _rows(self, x: torch.Tensor, B: int, what: str, trailing: tuple) -> torch.Tensor:
        """``x`` [1 or B, *trailing] (a name in ``trailing``: any size) on the device as B rows: one row is repeated."""
        if x.dim() != 1 + len(trailing) or x.shape[0] not in (1, B) or \
                any(isinstance(t, int) and n != t for n, t in zip(x.shape[1:], trailing)):
            dims = ", ".join(str(t) for t in trailing)
            raise ValueError(f"{what} must be [{'1' if B == 1 else f'1 or {B}'}, {dims}], got {tuple(x.shape)}")
        x = x.to(self.device)
        return x.repeat(B, *([1] * len(trailing))) if x.shape[0] < B else x

    @classmethod
    def random_init(cls, device="cuda", seed: int = 0, perturb_norm: bool = False, batch_invariant: bool = False) -> "TextToTimbre":
        """Deployed architecture (app.py:32-40) with deterministic synthetic weights (no checkpoints offline)."""
        unet = ConditionedUnet(**{k: v for k, v in W.UNET_DEPLOYED.items() if k not in ("out_dim", "time_dim")}, device=device,
                               batch_invariant=batch_invariant)
        unet.load_state_dict(W.unet_random_state_dict(seed=seed, perturb_norm=perturb_norm))
        vq = VQGAN(**W.VQGAN_DEPLOYED, device=device, batch_invariant=batch_invariant)
        vq.load_state_dict(W.vqgan_random_state_dict(seed=seed + 1, perturb_norm=perturb_norm))
        return cls(unet, vq, device=device)

    def sampler_for(self, batch: int, steps: int, cfg_scale: float, uncond: Optional[torch.Tensor]) -> DiffSynthSampler:
        """text2sound.py:96-106: fresh sampler, CFG activated, respaced to ``steps`` (cached per (batch, steps))."""
        return self._respaced_sampler((batch, steps), batch, steps, cfg_scale, uncond)

    def _respaced_sampler(self, key, batch: int, n_steps: int, cfg_scale: float, uncond: Optional[torch.Tensor],
                          noise_strategy: Optional[str] = None) -> DiffSynthSampler:
        """A sampler of ``batch`` rows respaced to ``n_steps`` as text2sound.py:96-106 builds it (``noise_strategy``: the pipeline's
        by default), cached under ``key``, with classifier-free guidance activated."""
        s = self._samplers.get(key)
        if s is None:
            s = DiffSynthSampler(self.timesteps, height=self.height, channels=self.channels, mute=True, device=str(self.device),
                                 max_batchsize=batch, noise_strategy=noise_strategy or self.noise_strategy)
            s.respace(list(np.linspace(0, self.timesteps - 1, n_steps, dtype=np.int32)))
            self._samplers[key] = s
        s.activate_classifier_free_guidance(cfg_scale, uncond)
        return s

    @torch.no_grad()
    def generate_from_tokens(self, text_encoder, input_ids: torch.Tensor, attention_mask: torch.Tensor, negative_ids: torch.Tensor,
                             negative_mask: torch.Tensor, **kw) -> Timbres:
        """text2sound.py:89-134 with the text front end on the device: ``text_encoder`` (diffusynth_b200.TextEncoder) turns the
        tokenizer's output for B DISTINCT prompts and for the one negative prompt into the condition / unconditional vectors
        (the reference encodes a single prompt on the CPU and repeats it, :89-91,109)."""
        cond = text_encoder.get_text_features(input_ids, attention_mask)
        uncond = text_encoder.get_text_features(negative_ids[:1], negative_mask[:1])[0]
        return self.generate(cond, uncond, **kw)

    @torch.no_grad()
    def generate(self, cond: torch.Tensor, uncond: Optional[torch.Tensor], steps: int = 20, cfg_scale: float = 6, width: int = 64,
                 sampler: str = "ddim", seed: Optional[int] = None, noise_feed: Optional[torch.Tensor] = None,
                 decode: bool = True) -> Timbres:
        """``noise_feed``: host or device draws [K, >=B, 4, 128, 64], draw 0 the initial noise and 1.. the per-step draws (K = 1:
        the initial noise only, e.g. ``[timbres.initial_noise]`` to re-create a timbre; later draws then come from the RNG).  The
        result's ``initial_noise`` is each row's train-width noise."""
        B = cond.shape[0]
        s = self.sampler_for(B, steps, cfg_scale, uncond)
        return self._run(s, lambda init: s.sample(self.unet, (B, self.channels, self.height, width), return_tensor=True,
                                                  condition=cond.to(self.device), sampler=sampler, initial_noise=init, seed=seed),
                         B, noise_feed, decode)

    # ---- timbre morphs (DiffSynthSampler.interpolate, model/DiffSynthSampler.py:224-269, from the pipeline) ------------------
    @torch.no_grad()
    def invert(self, latents: torch.Tensor, cond: torch.Tensor, uncond: Optional[torch.Tensor] = None, steps: int = 20,
               cfg_scale: float = 1.0) -> torch.Tensor:
        """DDIM inversion of latents [B,4,128,64] (e.g. encode_audio's) under their conditions [B, L]: the noises [B,4,128,64]
        from which generate / morph re-create them, in one graph launch for the batch (DiffSynthSampler.ddim_invert, a port
        extension).  The sampler is respaced to ``steps`` as generate's is (cached per batch and step count)."""
        if latents.dim() != 4 or tuple(latents.shape[1:]) != (self.channels, self.height, 64):
            raise ValueError(f"latents must be [B, {self.channels}, {self.height}, 64], got {tuple(latents.shape)}")
        B = latents.shape[0]
        if cond.dim() != 2 or cond.shape[0] != B:
            raise ValueError(f"cond must be [{B}, L], got {tuple(cond.shape)}")
        s = self._respaced_sampler(("invert", B, steps), B, steps, cfg_scale, uncond)
        s.final_only = True
        imgs, _ = s.ddim_invert(self.unet, latents, cond.to(self.device), return_tensor=True)
        self.last_launches = s.last_graph_launches
        return imgs[-1]

    def _morph_endpoints(self, first_noise, second_noise, first_cond, second_cond, frames, path):
        """Shape checks of morph (no device work): [P,4,128,64] / [4,128,64] noises and [P, L] / [L] conditions -> 4-D and 2-D views."""
        if self.noise_strategy != "repeat":
            raise ValueError(f"morph needs the 'repeat' noise strategy, not {self.noise_strategy!r}")
        if path not in MORPH_PATHS:
            raise ValueError(f"path must be one of {sorted(MORPH_PATHS)}, got {path!r}")
        if isinstance(frames, bool) or int(frames) != frames or frames < 2:
            raise ValueError(f"frames must be an integer >= 2, got {frames!r}")
        nz = (self.channels, self.height, 64)
        e = [x.unsqueeze(0) if x.dim() == 3 else x for x in (first_noise, second_noise)]
        c = [x.unsqueeze(0) if x.dim() == 1 else x for x in (first_cond, second_cond)]
        for x in e:
            if x.dim() != 4 or tuple(x.shape[1:]) != nz:
                raise ValueError(f"endpoint noises must be [P, {nz[0]}, {nz[1]}, {nz[2]}] or [{nz[0]}, {nz[1]}, {nz[2]}], got {tuple(x.shape)}")
        for x in c:
            if x.dim() != 2 or not x.is_floating_point():
                raise ValueError(f"endpoint conditions must be floating [P, L] or [L], got {tuple(x.shape)} {x.dtype}")
        if len({x.shape[0] for x in e + c}) != 1 or c[0].shape[1] != c[1].shape[1]:
            raise ValueError(f"endpoints disagree: noises {[tuple(x.shape) for x in e]}, conditions {[tuple(x.shape) for x in c]}")
        return e[0], e[1], c[0], c[1]

    @torch.no_grad()
    def morph(self, first_noise: torch.Tensor, second_noise: torch.Tensor, first_cond: torch.Tensor, second_cond: torch.Tensor,
              uncond: Optional[torch.Tensor], frames: int, path: str = "slerp", steps: int = 20, cfg_scale: float = 6, width: int = 64,
              sampler: str = "ddim", seed: Optional[int] = None, decode: bool = True) -> Timbres:
        """P timbre morphs of ``frames`` frames each: frame k of sequence p starts from the noise between first_noise[p] and
        second_noise[p] at a = k / (frames - 1) (``path`` "slerp", or "linear" = the reference's interpolate) under the linearly
        interpolated condition, and the P * frames rows sample with classifier-free guidance and decode through the usual VQ ->
        decoder -> iSTFT tail in ONE graph launch.  Endpoint noises are train-width noises [P,4,128,64] (``Timbres.initial_noise``
        of generate, or invert of an upload); a [4,128,64] noise / [L] condition is P = 1.  Rows are sequence-major; the result's
        initial_noise holds the rows' noises."""
        e0, e1, c0, c1 = self._morph_endpoints(first_noise, second_noise, first_cond, second_cond, frames, path)
        dev = self.device
        noise, cond = morph_rows(e0.to(dev), e1.to(dev), c0.to(dev), c1.to(dev), int(frames), path)      # one ds_morph_rows
        rows = noise.view(1, noise.shape[0], self.channels, self.height, 64)
        return self.generate(cond, uncond, steps=steps, cfg_scale=cfg_scale, width=width, sampler=sampler, seed=seed, noise_feed=rows,
                             decode=decode)


    # ---- timbre modification (sound2sound_with_text.py:47-269) -------------------------------------------------------
    @torch.no_grad()
    def encode_audio(self, wave, width: int = 64, sample_rate=16000) -> torch.Tensor:
        """receive_upload_origin_audio's tensor path (:75-107): peak-normalise, resample to 16 kHz and crop/zero-pad to
        256*(4w-1) samples (adjust_audio_length, :80-82), STFT (1024/256, hann) -> pad_STFT -> encode_stft -> VQGAN encoder.
        ``wave``: a [B, L] tensor / array, or a list of 1-D clips of different lengths; ``sample_rate``: an integer, or one per
        clip.  Normalisation, resampling and the length adjustment are one ds_resample call writing the STFT's input (a 16 kHz clip
        is copied).  Returns the UN-quantised latent [B,4,128,w] (:107)."""
        if isinstance(wave, (list, tuple)):
            if not wave or any(np.ndim(c) != 1 for c in wave):
                raise ValueError("expected a non-empty list of 1-D clips")
        elif np.ndim(wave) != 2:
            raise ValueError("expected a [B, L] batch or a list of 1-D clips")
        parts, shapes, _ = _layout(wave, 1)
        B, n = len(shapes), 256 * (4 * width - 1)
        wave = resample_packed(_pack(parts, self.device), [L for L, in shapes], sample_rate, SAMPLE_RATE, out_lengths=n,
                               normalize_peak=True).view(B, n)                                             # :75-82
        # pad_STFT(D) is called with its default time_resolution = 256 frames and never crops (tools.py:170-182): clips of
        # <= 3 s (width <= 64) always encode to a 64-column latent, longer ones to ``width`` columns
        spec = waveform_to_spectrogram(wave, time_resolution=max(256, 4 * width))          # :85-94
        return self.vqgan._encoder(spec)

    @torch.no_grad()
    def modify(self, guide_latent: torch.Tensor, cond: torch.Tensor, uncond: Optional[torch.Tensor], steps: int = 20,
               strength: float = 0.7, cfg_scale: float = 6, sampler: str = "ddim", seed: Optional[int] = None,
               noise_feed: Optional[torch.Tensor] = None, decode: bool = True) -> Timbres:
        """sound2sound_sample (:126-269): respace to int(steps/strength) (:185), img_guided_sample(noising_strength=strength,
        guide_img=latent.repeat(B)) (:194-203), then the same VQ -> decoder -> iSTFT tail as text-to-timbre."""
        B = cond.shape[0]
        guide = self._rows(guide_latent, B, "guide_latent", (self.channels, self.height, "w")).float()
        width = guide.shape[-1]
        n_steps = int(steps / strength)
        s = self._respaced_sampler(("modify", B, n_steps), B, n_steps, cfg_scale, uncond)
        return self._run(s, lambda init: s.img_guided_sample(self.unet, (B, self.channels, self.height, width), strength, guide,
                                                             return_tensor=True, condition=cond.to(self.device), sampler=sampler,
                                                             initial_noise=init, seed=seed),
                         B, noise_feed, decode)

    # ---- inpainting with text (inpaint_with_text.py:140-333) ----------------------------------------------------------
    @torch.no_grad()
    def inpaint(self, guide_latent: torch.Tensor, mask, cond: torch.Tensor, uncond: Optional[torch.Tensor], steps: int = 20,
                cfg_scale: float = 6, noising_strength: float = 1.0, sampler: str = "ddim", seed: Optional[int] = None,
                noise_feed: Optional[torch.Tensor] = None, decode: bool = True) -> Timbres:
        """Regenerate the masked part of an upload from text: the mask is zoomed to the latent grid (scipy.ndimage.zoom with its
        defaults, no threshold), then inpaint_sample with classifier-free guidance (:229-231) and the same VQ -> decoder -> iSTFT
        tail as text-to-timbre, in one graph launch for the whole batch.
        ``guide_latent``: [1 or B, 4, 128, w], e.g. from encode_audio.  ``mask``: 1 keeps the upload, 0 regenerates; in the
        spectrogram's orientation (row 0 = lowest frequency, last axis = time; flip an image-oriented mask first) on any grid,
        e.g. 513 x T as InputBatch2Encode_STFT renders it after np.flipud, or 512 x 4w; one 2-D array / tensor for every row, a
        [B, H, W] one, or a list of B 2-D ones of any shapes.  All masks go through ONE ds_mask_zoom into the [B, 1, 128, w]
        mask the sampling graph reads.  The sampler is respaced to ``steps`` (cached per (batch, steps)), as generate does."""
        B = cond.shape[0]
        guide = self._rows(guide_latent, B, "guide_latent", (self.channels, self.height, "w")).float()
        width = guide.shape[-1]
        if isinstance(mask, (list, tuple)):
            if len(mask) != B or any(np.ndim(m) != 2 for m in mask):
                raise ValueError(f"a list mask must hold {B} 2-D arrays")
        elif not (np.ndim(mask) == 2 or np.ndim(mask) == 3 and np.shape(mask)[0] == B):
            raise ValueError(f"mask must be 2-D, [{B}, H, W] or a list of {B} 2-D arrays, got shape {tuple(np.shape(mask))}")
        parts, shapes, _ = _layout(mask, 2)
        zoomed = torch.empty((len(shapes), 1, self.height, width), dtype=torch.float32, device=self.device)
        zoom_packed(_pack(parts, self.device), shapes, (self.height, width), out=zoomed)
        s = self._respaced_sampler(("inpaint", B, steps), B, steps, cfg_scale, uncond)
        return self._run(s, lambda init: s.inpaint_sample(self.unet, (B, self.channels, self.height, width), noising_strength, guide,
                                                          zoomed, return_tensor=True, condition=cond.to(self.device), sampler=sampler,
                                                          initial_noise=init, seed=seed),
                         B, noise_feed, decode)


    # ---- per-note synthesis for arrangements (track_maker.py:228-283) ---------------------------------------------------
    @staticmethod
    def note_width(duration_sec: float, time_resolution: int = 256, vae_scale: int = 4) -> int:
        return int(time_resolution * ((duration_sec + 1) / 4) / vae_scale)                                    # track_maker.py:245

    @torch.no_grad()
    def synthesize_note(self, instrument_latent: torch.Tensor, condition: torch.Tensor, duration_sec: float, sample_steps: int = 20,
                        noising_strength: float = 1.0, attack: float = 0.5, before_release: float = 0.5, sampler: str = "ddim",
                        time_resolution: int = 256, vae_scale: int = 4, noise_feed: Optional[torch.Tensor] = None) -> Timbres:
        """One note of an instrument at an arbitrary duration: the ``diffSynthSampler`` closure of track_maker.DiffSynth.
        ``instrument_latent`` [1,4,128,64] is the instrument's latent (re-laid to the note's width by the repeat strategy),
        ``condition`` [1,512] the empty-prompt embedding the reference passes (:231-233; no classifier-free guidance here);
        attack and tail are frozen by a mask that shrinks over the steps (``use_dynamic_mask``, mask_flexivity 1.0).
        The width ``int(256 * ((duration + 1) / 4) / 4)`` is arbitrary, odd levels included (pad_to_match)."""
        return self.synthesize_notes(instrument_latent, condition, [duration_sec], sample_steps, noising_strength, attack, before_release,
                                     sampler, time_resolution, vae_scale, None if noise_feed is None else [noise_feed])[0]

    @torch.no_grad()
    def synthesize_notes(self, instrument_latent: torch.Tensor, condition: torch.Tensor, durations_sec, sample_steps: int = 20,
                         noising_strength: float = 1.0, attack: float = 0.5, before_release: float = 0.5, sampler: str = "ddim",
                         time_resolution: int = 256, vae_scale: int = 4, noise_feeds=None) -> list:
        """The notes of a track (track_maker.py:285-330 calls the per-note closure once per distinct duration): notes of equal
        duration -- hence equal latent width -- are batched into ONE graph launch (SURVEY 8f item 1).  Returns one ``Timbres`` per
        note, in input order.  ``noise_feeds`` (tests): per note a host noise tensor [count, 1, C, H, 64]."""
        widths = [self.note_width(d, time_resolution, vae_scale) for d in durations_sec]
        return self._synthesize_rows([instrument_latent] * len(widths), [condition] * len(widths), widths, sample_steps, noising_strength,
                                     attack, before_release, sampler, time_resolution, vae_scale, noise_feeds)

    def _synthesize_rows(self, latents, conditions, widths, sample_steps, noising_strength, attack, before_release, sampler, time_resolution,
                         vae_scale, noise_feeds) -> list:
        """Rows of equal width -- whatever their instrument latent [1,4,128,64] and condition [1,512] -- as ONE batched inpainting
        run (one graph launch) per distinct width: every row is an independent sample of the batch (own guide, condition and noise
        rows), exactly what separate calls of the reference's per-note closure compute.  Returns one ``Timbres`` per row, in order;
        ``noise_feeds``: None or one per row."""
        out = [None] * len(widths)
        for w in sorted(set(widths)):
            idx = [i for i, ww in enumerate(widths) if ww == w]
            B = len(idx)
            guide = torch.cat([self._rows(latents[i], 1, "instrument_latent", (self.channels, self.height, 64)) for i in idx]).float()
            cond = torch.cat([self._rows(conditions[i], 1, "condition", ("L",)) for i in idx])
            feed = None if noise_feeds is None else noise_feeds[idx[0]] if B == 1 else torch.cat([noise_feeds[i] for i in idx], dim=1)
            # the reference builds a fresh sampler per note (:248-249); here it is cached per (step count, batch) so that the captured
            # graph of a (width, steps, batch) triple is reused by every later group of that shape instead of being re-captured
            s = self._respaced_sampler(("note", sample_steps, B), B, sample_steps, 1.0, None, noise_strategy="repeat")
            mask = torch.zeros((B, 1, self.height, w), dtype=torch.float32, device=self.device)                # :252-254
            mask[:, :, :, :int(time_resolution * (attack / 4) / vae_scale)] = 1.0
            mask[:, :, :, -int(time_resolution * ((before_release + 1) / 4) / vae_scale):] = 1.0
            # :257-269, then the quantiser (:275), decoder and iSTFT (:277-283) inside the group's graph
            t = self._run(s, lambda init: s.inpaint_sample(self.unet, (B, self.channels, self.height, w), noising_strength, guide, mask,
                                                           return_tensor=True, condition=cond, sampler=sampler, initial_noise=init,
                                                           use_dynamic_mask=True, end_noise_level_ratio=0.0, mask_flexivity=1.0),
                          B, feed, True)
            for b, i in enumerate(idx):
                out[i] = Timbres(t.latents[b:b + 1], t.quantized[b:b + 1], t.spectrograms[b:b + 1], t.waveforms[b:b + 1],
                                 t.initial_noise[b:b + 1])
        return out

    @staticmethod
    def track_plan(notes, time_resolution: int = 256, vae_scale: int = 4, sample_rate: int = 16000) -> TrackPlan:
        """Host side of render_track: notes ``(onset_sec, duration_sec, semitones, gain)`` -> the distinct durations and the distinct
        (duration, semitones) pairs in order of first appearance, each note's pair, onsets in samples (round(onset * 16000)), note
        lengths in samples and the track length."""
        durations, pairs, note_pair, onsets, gains, lengths = [], [], [], [], [], []
        for onset_sec, dur, semi, gain in notes:
            dur, semi = float(dur), float(semi)
            if dur not in durations:
                durations.append(dur)
            key = (durations.index(dur), semi)
            if key not in pairs:
                pairs.append(key)
            note_pair.append(pairs.index(key))
            onsets.append(int(round(float(onset_sec) * sample_rate)))
            gains.append(float(gain))
            lengths.append(256 * (4 * TextToTimbre.note_width(dur, time_resolution, vae_scale) - 1))
            if onsets[-1] < 0:
                raise ValueError(f"note onsets must be >= 0, got {onset_sec}")
        track_len = max(o + n for o, n in zip(onsets, lengths))
        return TrackPlan(durations, pairs, note_pair, onsets, gains, lengths, track_len)

    @torch.no_grad()
    def render_track(self, instrument_latent: torch.Tensor, condition: torch.Tensor, notes, sample_steps: int = 20,
                     noising_strength: float = 1.0, attack: float = 0.5, before_release: float = 0.5, sampler: str = "ddim",
                     time_resolution: int = 256, vae_scale: int = 4, noise_feeds=None) -> torch.Tensor:
        """A note arrangement rendered on the device: what track_maker.DiffSynth does after its per-note closure.  ``notes`` is a
        list of ``(onset_sec, duration_sec, semitones, gain)``.  One timbre is synthesised per distinct duration (synthesize_notes,
        same keyword arguments; ``noise_feeds``: one per distinct duration, in order of first appearance), each distinct
        (duration, semitones) pair is pitch-shifted once (librosa.effects.pitch_shift, track_maker.py:42) in one batched call, and
        every note is placed at round(onset * 16000) with its gain and summed in one call (codec.shift_and_mix).  Returns the
        fp32 track [max(onset + note length)]; no normalisation, no envelope."""
        return self._render([(instrument_latent, condition, notes, 1.0, 0.0)], sample_steps, noising_strength, attack, before_release,
                            sampler, time_resolution, vae_scale, noise_feeds, fades=False, target_peak=None)

    @staticmethod
    def arrangement_plan(tracks, time_resolution: int = 256, vae_scale: int = 4, sample_rate: int = 16000,
                         reverb_sends=None) -> ArrangementPlan:
        """Host side of render_arrangement: ``tracks`` of ``(instrument_latent, condition, notes, gain, fade_out_sec[, pan])`` ->
        track_plan per track, joined: the synthesis rows (one per distinct (track, duration)) and their widths, the pitch items (one
        per distinct (row, semitones)), and per note in mix order (tracks in order, notes in order) its item, onset, gain (note gain *
        track gain), fade (round(fade_out_sec * 16000) samples), pan (the track's, 0 without one), reverb send (reverb_sends[track],
        one finite value >= 0 per track; 1.0 when None) and length; the track length is the end of the last note."""
        if len(tracks) == 0:
            raise ValueError("an arrangement needs at least one track")
        track_sends = [1.0] * len(tracks) if reverb_sends is None else [float(v) for v in _check_sends(reverb_sends, len(tracks))]
        rows, widths, items, note_item, onsets, gains, fades, pans, sends, lengths = [], [], [], [], [], [], [], [], [], []
        for k, track in enumerate(tracks):
            if len(track) not in (5, 6):
                raise ValueError(f"track {k}: expected (instrument_latent, condition, notes, gain, fade_out_sec[, pan]), got "
                                 f"{len(track)} fields")
            _, _, notes, gain, fade_sec = track[:5]
            pan = float(track[5]) if len(track) == 6 else 0.0
            if len(notes) == 0:
                raise ValueError(f"track {k} has no notes")
            if not np.isfinite(float(fade_sec)) or float(fade_sec) < 0:
                raise ValueError(f"track {k}: fade_out_sec must be finite and >= 0, got {fade_sec}")
            if not np.isfinite(pan) or abs(pan) > 1:
                raise ValueError(f"track {k}: pan must be finite and in [-1, 1], got {track[5]}")
            fade = int(round(float(fade_sec) * sample_rate))
            p = TextToTimbre.track_plan(notes, time_resolution, vae_scale, sample_rate)
            r0, i0 = len(rows), len(items)
            rows += [(k, d) for d in p.durations]
            widths += [TextToTimbre.note_width(d, time_resolution, vae_scale) for d in p.durations]
            items += [(r0 + d, semi) for d, semi in p.pairs]
            note_item += [i0 + i for i in p.note_pair]
            onsets += p.onsets
            gains += [g * float(gain) for g in p.gains]
            fades += [fade] * len(p.onsets)
            pans += [pan] * len(p.onsets)
            sends += [track_sends[k]] * len(p.onsets)
            lengths += p.lengths
        track_len = max(o + n for o, n in zip(onsets, lengths))
        return ArrangementPlan(rows, widths, items, note_item, onsets, gains, fades, lengths, track_len, pans, sends)

    @torch.no_grad()
    def render_arrangement(self, tracks, sample_steps: int = 20, noising_strength: float = 1.0, attack: float = 0.5,
                           before_release: float = 0.5, sampler: str = "ddim", target_peak: Optional[float] = None,
                           time_resolution: int = 256, vae_scale: int = 4, noise_feeds=None, stereo: bool = False,
                           impulse_response=None, reverb_sends=None) -> torch.Tensor:
        """Several instruments rendered into one piece on the device: track_maker.DiffSynth over several Tracks, summed.  ``tracks``
        is a list of ``(instrument_latent [1,4,128,64], condition [1,512], notes, gain, fade_out_sec)``, ``notes`` as render_track
        takes them.  The (track, duration) rows of ALL tracks are synthesised with one graph launch per distinct width, each row
        with its own instrument latent and condition; every distinct (row, semitones) item is pitch-shifted in one call; every note
        is placed with its gain times its track's gain, faded out linearly over the last fade_out_sec of its waveform, and summed
        in one call (ds_mix_arrangement).  ``target_peak``: None, or max |result| after a peak normalisation on the device, a
        finite value > 0 (codec._check_peak, before any synthesis).  ``noise_feeds`` (tests): one per row (arrangement_plan), in row
        order.  Returns the fp32 piece [max(onset + note length)].

        ``stereo=True`` mixes into two channels instead (ds_mix_stereo) and returns the planar [2, max(onset + note length)], left
        then right.  A track may then carry a sixth field, its pan in [-1, 1] (-1 left, 0 centre, 1 right; a 5-tuple track is
        centred), applied to each of its notes with a constant-power law (codec.mix_stereo); ``target_peak`` scales both channels
        by one factor.  With ``stereo=False`` a 6-tuple track is an error.

        ``impulse_response`` adds convolution reverb (codec.shift_and_mix): a 16 kHz impulse response [M], or with ``stereo=True``
        [2, M] (left, right), as a host or device tensor or a numpy array, used as given, so its level is the wet level.  An IR
        recorded at another rate is converted first with codec.resample(ir, sr, 16000).  ``reverb_sends``: one finite send level
        >= 0 per track (None: 1.0 for every track; an error without an IR).  The send is post-fader and post-pan: the send bus is
        every note with its gain times its track's send, with the same fades and pans.  The result is dry + IR * bus, the piece
        followed by the reverb tail: [L + M - 1], or planar [2, L + M - 1] in stereo, L = max(onset + note length).  A mono IR
        convolves both channels of a stereo piece; a [2, M] IR convolves left with left and right with right.  ``target_peak``
        applies after the reverb is added, with one factor over both channels.  Every argument is checked before synthesis."""
        _check_peak(target_peak)
        if not stereo and any(len(t) == 6 for t in tracks):
            raise ValueError("a track with a pan (6 fields) needs stereo=True")
        if impulse_response is None and reverb_sends is not None:
            raise ValueError("reverb_sends needs an impulse_response")
        if reverb_sends is not None:
            _check_sends(reverb_sends, len(tracks))
        ir = None if impulse_response is None else _check_impulse_response(impulse_response, stereo)
        return self._render(tracks, sample_steps, noising_strength, attack, before_release, sampler, time_resolution, vae_scale,
                            noise_feeds, fades=True, target_peak=target_peak, stereo=stereo, impulse_response=ir,
                            reverb_sends=reverb_sends)

    def _render(self, tracks, sample_steps, noising_strength, attack, before_release, sampler, time_resolution, vae_scale, noise_feeds,
                fades: bool, target_peak: Optional[float], stereo: bool = False, impulse_response: Optional[torch.Tensor] = None,
                reverb_sends=None) -> torch.Tensor:
        """render_arrangement's body: the plan, one synthesis launch per distinct width, one pitch shift and one mix.  ``fades``
        False (render_track) mixes through ds_mix_track, without the tracks' fades; ``stereo`` through ds_mix_stereo; a checked
        ``impulse_response`` [H, M] adds a second mix (the send bus) and one convolution."""
        plan = self.arrangement_plan(tracks, time_resolution, vae_scale, reverb_sends=reverb_sends)
        latents, conditions = [], []
        for k, (lat, cond) in enumerate(t[:2] for t in tracks):
            if tuple(lat.shape) != (1, self.channels, self.height, 64):
                raise ValueError(f"track {k}: instrument_latent must be [1, {self.channels}, {self.height}, 64], got {tuple(lat.shape)}")
            if cond.dim() != 2 or cond.shape[0] != 1:
                raise ValueError(f"track {k}: condition must be [1, L], got {tuple(cond.shape)}")
            latents.append(lat)
            conditions.append(cond)
        if len({c.shape[1] for c in conditions}) != 1:
            raise ValueError("every track's condition must have the same length")
        timbres = self._synthesize_rows([latents[k] for k, _ in plan.rows], [conditions[k] for k, _ in plan.rows], plan.widths,
                                        sample_steps, noising_strength, attack, before_release, sampler, time_resolution, vae_scale,
                                        noise_feeds)
        sources = [timbres[r].waveforms[0] for r, _ in plan.items]
        track = shift_and_mix(sources, [s for _, s in plan.items], plan.note_item, plan.onsets, plan.gains,
                              fades=plan.fades if fades else None, target_peak=target_peak, pans=plan.pans if stereo else None,
                              impulse_response=impulse_response, sends=plan.sends)
        assert track.shape[-1] == plan.track_len + (0 if impulse_response is None else impulse_response.shape[1] - 1)
        return track


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous split of ``total`` prompts: rank r owns [lo, hi); per = ceil(total/world)."""
    per = -(-total // world)
    lo = min(rank * per, total)
    return lo, min(lo + per, total)


def all_gather_waveforms(local: torch.Tensor, total: int, world: int) -> torch.Tensor:
    """One equal-count all-gather of [per, L] waveforms (NCCL on GPUs, gloo in CPU tests) -> [total, L] on every rank."""
    import torch.distributed as dist
    per = -(-total // world)
    if local.shape[0] < per:
        local = torch.cat([local, local.new_zeros((per - local.shape[0],) + tuple(local.shape[1:]))])
    out = local.new_empty((world * per,) + tuple(local.shape[1:]))
    dist.all_gather_into_tensor(out, local.contiguous())
    return out[:total]


class ChunkGatherer:
    """The collective half of the sharded job: rank-local result chunks [chunk, L] are all-gathered one by one (NCCL on a side
    stream on GPUs, so that chunk k travels while chunk k+1 is computed; gloo / plain copies on CPU tensors in the host tests) into
    the rank-major result [world, per_pad, L]; ``finish()`` returns the first ``total`` rows in prompt order."""

    def __init__(self, total: int, rank: int, world: int, chunk: int, L: int, device, dtype=torch.float32, comm=None):
        self.total, self.rank, self.world, self.chunk, self.L = total, rank, world, chunk, L
        self.comm_handle = comm      # engine.Comm (the library's own NCCL communicator, ds_allgather) or None = torch.distributed
        self.per = -(-total // world)
        self.n_chunks = -(-self.per // chunk)
        self.device = torch.device(device)
        self.cuda = self.device.type == "cuda"
        self.comm = torch.cuda.Stream(device=self.device) if self.cuda else None
        self.out = torch.zeros((world, self.n_chunks * chunk, L), dtype=dtype, device=self.device)
        self.stage = [torch.empty((world, chunk, L), dtype=dtype, device=self.device) for _ in range(2)]
        self._exposed = None

    def submit(self, k: int, w: torch.Tensor) -> None:
        """Chunk k of this rank (rows past the rank's share zero-padded by the caller to [chunk, L])."""
        import torch.distributed as dist
        assert tuple(w.shape) == (self.chunk, self.L), tuple(w.shape)

        def gather():
            if self.world > 1:
                st = self.stage[k % 2]
                if self.comm_handle is not None:
                    self.comm_handle.all_gather(w, recv=st.view(self.world * self.chunk, self.L))
                else:
                    dist.all_gather_into_tensor(st.view(self.world * self.chunk, self.L), w.contiguous())
                self.out[:, k * self.chunk:(k + 1) * self.chunk].copy_(st)
            else:
                self.out[0, k * self.chunk:(k + 1) * self.chunk].copy_(w)

        if not self.cuda:
            gather()
            return
        main = torch.cuda.current_stream(self.device)
        ready = torch.cuda.Event()
        ready.record(main)
        with torch.cuda.stream(self.comm):
            self.comm.wait_event(ready)
            gather()
            w.record_stream(self.comm)

    def finish(self) -> torch.Tensor:
        if self.cuda:
            main = torch.cuda.current_stream(self.device)
            t_main, t_comm = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_main.record(main)
            t_comm.record(self.comm)
            main.wait_stream(self.comm)
            self._exposed = (t_main, t_comm)
        return self.out[:, :self.per].reshape(self.world * self.per, self.L)[:self.total]

    def exposed_ms(self) -> float:
        """How long the side stream ran past the end of the last chunk's compute in the most recent job (synchronises)."""
        if self._exposed is None:
            return 0.0
        t_main, t_comm = self._exposed
        t_comm.synchronize()
        return max(0.0, t_main.elapsed_time(t_comm))


class ShardedGenerator:
    """BASELINE configs[3] / SURVEY 8(e): ``total`` prompts split contiguously over ``world`` ranks; each rank samples its share in
    chunks of ``chunk`` prompts through the text-to-timbre graph and the waveforms of chunk k are all-gathered on a side stream
    while chunk k+1 is being sampled, so that only the last chunk's gather is exposed.  Every rank ends with all waveforms
    [total, L] in prompt order."""

    def __init__(self, pipe: TextToTimbre, total: int, rank: int, world: int, chunk: int = 64, comm=None):
        self.pipe, self.total, self.rank, self.world, self.chunk = pipe, total, rank, world, chunk
        self.comm = comm
        self.lo, self.hi = shard_range(total, rank, world)
        self.gatherer: Optional[ChunkGatherer] = None
        self.n_chunks = -(-(-(-total // world)) // chunk)
        self.launches_per_job = 0

    @torch.no_grad()
    def run(self, cond: torch.Tensor, uncond: Optional[torch.Tensor], steps: int = 20, cfg_scale: float = 6, width: int = 64,
            sampler: str = "ddim", seed: Optional[int] = None) -> torch.Tensor:
        pipe, chunk = self.pipe, self.chunk
        L = 256 * (4 * width - 1)
        if self.gatherer is None or self.gatherer.L != L:
            self.gatherer = ChunkGatherer(self.total, self.rank, self.world, chunk, L, pipe.device, comm=self.comm)
        n_local = self.hi - self.lo
        launches = 0
        for k in range(self.n_chunks):
            c = cond[k * chunk:min((k + 1) * chunk, n_local)]
            if c.shape[0] > 0:
                w = pipe.generate(c, uncond, steps=steps, cfg_scale=cfg_scale, width=width, sampler=sampler, seed=seed).waveforms
                launches += pipe.last_launches
                if w.shape[0] < chunk:
                    w = torch.cat([w, w.new_zeros((chunk - w.shape[0], L))])
            else:
                w = torch.zeros((chunk, L), dtype=torch.float32, device=pipe.device)       # (a rank past the end of the prompt list)
            self.gatherer.submit(k, w)
        self.launches_per_job = launches
        return self.gatherer.finish()

    def exposed_gather_ms(self) -> float:
        return self.gatherer.exposed_ms() if self.gatherer is not None else 0.0
