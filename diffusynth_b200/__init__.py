"""diffusynth_b200 -- B200 (sm_100a) implementation of DiffuSynth's text-to-timbre sampling path.

Python surfaces mirror the reference (WxuanYuan/diffusynth): ``DiffSynthSampler``, ``ConditionedUnet``,
``VQGAN`` / ``VectorQuantizerEMA`` / ``Decoder`` / ``Encoder``, and the spectrogram <-> waveform transforms;
the arithmetic runs in hand-written CUDA kernels behind the C ABI of ``include/diffusynth_b200.h``.
Importing the compute classes needs a CUDA build of torch; there is no CPU fallback."""
from . import weights  # noqa: F401  (pure-python parameter inventory; safe everywhere)

__all__ = ["weights", "DiffSynthSampler", "ConditionedUnet", "VQGAN", "VectorQuantizerEMA", "Decoder", "Encoder",
           "TextToTimbre", "TextEncoder", "spectrogram_to_waveform", "waveform_to_spectrogram", "pitch_shift", "mix_track", "mix_arrangement",
           "mix_stereo", "fftconvolve", "morph_rows"]


def __getattr__(name):
    if name == "DiffSynthSampler":
        from .sampler import DiffSynthSampler
        return DiffSynthSampler
    if name == "ConditionedUnet":
        from .unet import ConditionedUnet
        return ConditionedUnet
    if name in ("VQGAN", "VectorQuantizerEMA", "Decoder", "Encoder"):
        from . import vqgan
        return getattr(vqgan, name)
    if name == "TextEncoder":
        from .text import TextEncoder
        return TextEncoder
    if name == "TextToTimbre":
        from .pipeline import TextToTimbre
        return TextToTimbre
    if name in ("spectrogram_to_waveform", "waveform_to_spectrogram", "encodeBatch2GradioOutput_STFT", "InputBatch2Encode_STFT",
                "spectrogram_images", "latent_images", "latent_representation_to_Gradio_image", "griffinlim",
                "pitch_shift", "mix_track", "mix_arrangement", "mix_stereo", "shift_and_mix", "fftconvolve", "morph_rows"):
        from . import codec
        return getattr(codec, name)
    raise AttributeError(name)
