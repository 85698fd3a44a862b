"""ctypes binding of libdiffusynth_b200.so (the C ABI declared in include/diffusynth_b200.h).

There is NO CPU fallback: if the shared library is missing or does not load, importing any
compute entry point raises.  ``load()`` builds the library in-tree when nvcc is available
and the sources are newer than the binary."""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DS_LIB_PATH") or os.path.join(HERE, "libdiffusynth_b200.so")   # DS_LIB_PATH: A/B builds (tools_dev)
HEADER = os.path.join(os.path.dirname(HERE), "include", "diffusynth_b200.h")

DS_MAX_TAPS = 16
DS_MAX_GROUPS = 4


class ConvTap(C.Structure):
    _fields_ = [("dy", C.c_int8), ("dx", C.c_int8), ("view", C.c_int8), ("pad_", C.c_int8)]


class ConvGemmArgs(C.Structure):
    _fields_ = [
        ("d_src0", C.c_void_p), ("d_src1", C.c_void_p),
        ("C0", C.c_int32), ("C1", C.c_int32), ("N", C.c_int32), ("src_batch_mod", C.c_int32),
        ("Hv", C.c_int32), ("Wv", C.c_int32),
        ("view_sn", C.c_int64), ("view_sh", C.c_int64), ("view_sw", C.c_int64),
        ("view_off", C.c_int64 * 4), ("num_views", C.c_int32),
        ("view_wv", C.c_int32 * 4), ("view_hv", C.c_int32 * 4),
        ("H", C.c_int32), ("W", C.c_int32), ("Hb", C.c_int32), ("Wb", C.c_int32),
        ("d_weight", C.c_void_p),
        ("Cout_pad", C.c_int32), ("Cout", C.c_int32), ("BN", C.c_int32), ("BK", C.c_int32),
        ("ntaps", C.c_int32), ("groups", C.c_int32), ("per_sample_weights", C.c_int32),
        ("taps", (ConvTap * DS_MAX_TAPS) * DS_MAX_GROUPS),
        ("d_stats_in", C.c_void_p), ("stats_in_slots", C.c_int32), ("stats_out_inv_count", C.c_float), ("eps", C.c_float),
        ("d_e1", C.c_void_p), ("d_e2", C.c_void_p), ("ncls", C.c_int32),
        ("d_sbias", C.c_void_p), ("sbias_stride", C.c_int32), ("act", C.c_int32),
        ("d_residual", C.c_void_p), ("res_sn", C.c_int64), ("res_sh", C.c_int64), ("res_sw", C.c_int64),
        ("d_out", C.c_void_p), ("out_sn", C.c_int64), ("out_sh", C.c_int64), ("out_sw", C.c_int64),
        ("out_goff", C.c_int64 * DS_MAX_GROUPS),
        ("d_out_f32_nchw", C.c_void_p), ("d_stats_out", C.c_void_p),
    ]


class ConvGemmPlanInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("BK", "BN", "cg", "pair_flat", "epi", "two_per_sm", "nacc", "sps", "stages", "num_tiles", "grid")]


_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_longlong, C.c_float
_SIGNATURES = {
    "ds_last_error": (C.c_char_p, []),
    "ds_version": (_I, []),
    "ds_operand_dtype": (_I, []),
    "ds_check_device": (_I, [_I]),
    "ds_conv_gemm": (_I, [C.POINTER(ConvGemmArgs), _P]),
    "ds_conv_gemm_reference": (_I, [C.POINTER(ConvGemmArgs), _P]),
    "ds_conv_gemm_stats_slots": (_I, [C.POINTER(ConvGemmArgs)]),
    "ds_conv_gemm_plan": (_I, [C.POINTER(ConvGemmArgs), C.POINTER(ConvGemmPlanInfo)]),
    "ds_ddim_step": (_I, [_P, _P, _P, _P, _P, _P, _L, _P]),
    "ds_q_sample": (_I, [_P, _P, _P, _P, _L, _L, _P]),
    "ds_mask_blend": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _L, _P]),
    "ds_dwconv7": (_I, [_P, _P, _I, _I, _I, _P, _P, _L, _P, _P, _F, _I, _I, _I, _P]),
    "ds_dwconv7_stats_slots": (_I, [_I, _I, _I]),
    "ds_stem_im2col": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "ds_sinusoidal_embedding": (_I, [_P, _P, _I, _I, _P]),
    "ds_embedding_gather": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "ds_linear": (_I, [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _I, _P]),
    "ds_attn_chunks": (_I, [_L]),
    "ds_attn_part_floats": (_L, [_I, _I, _L]),
    "ds_attn_ctx_partial": (_I, [_P, _P, _P, _I, _I, _L, _I, _F, _P]),
    "ds_attn_qkv_ctx": (_I, [_P, _I, _I, _P, _I, _P, _P, _P, _P, _L, _P, _P, _I, _I, _L, _F, _P]),
    "ds_attn_finalize": (_I, [_P, _P, _P, _I, _I, _L, _I, _I, _P]),
    "ds_attn_finalize_cat": (_I, [_P, _P, _P, _L, _P, _P, _I, _I, _L, _I, _I, _P]),
    "ds_gn_apply_residual": (_I, [_P, _P, _P, _P, _I, _P, _P, _I, _I, _L, _I, _P]),
    "ds_vq_quantize": (_I, [_P, _P, _I, _P, _P, _I, _L, _P]),
    "ds_group_stats": (_I, [_P, _P, _I, _I, _I, _I, _L, _I, _P]),
    "ds_gn_act": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _L, _F, _I, _P]),
    "ds_add_bf16": (_I, [_P, _P, _P, _L, _P]),
    "ds_add_channel_bias": (_I, [_P, _P, _L, _I, _I, _L, _P]),
    "ds_decoder_head": (_I, [_P, _P, _P, _I, _L, _P]),
    "ds_nchw_f32_to_nhwc_bf16": (_I, [_P, _P, _I, _I, _I, _L, _P]),
    "ds_nhwc_bf16_to_nchw_f32": (_I, [_P, _P, _I, _I, _I, _L, _P]),
    "ds_istft_length": (_L, [_I]),
    "ds_stft_decode_istft": (_I, [_P, _P, _P, _I, _I, _P]),
    "ds_stft_encode": (_I, [_P, _L, _P, _I, _I, _P]),
    "ds_decode_stft": (_I, [_P, _P, _L, _I, _P]),
    "ds_encode_stft": (_I, [_P, _P, _L, _I, _P]),
    "ds_griffinlim_update": (_I, [_P, _P, _P, _F, _I, _I, _I, _P]),
    "ds_pitch_shift_workspace": (_I, [_P, _P, _I, _P, _P]),
    "ds_pitch_shift": (_I, [_P, _P, _P, _P, _I, _P, _L, _P]),
    "ds_mix_track_workspace": (_I, [_P, _P, _I, _L, _P]),
    "ds_mix_track": (_I, [_P, _P, _P, _P, _P, _I, _P, _L, _P, _L, _P]),
    "ds_mix_arrangement_workspace": (_I, [_P, _P, _P, _I, _F, _L, _P]),
    "ds_mix_arrangement": (_I, [_P, _P, _P, _P, _P, _P, _I, _F, _P, _L, _P, _L, _P]),
    "ds_mix_stereo_workspace": (_I, [_P, _P, _P, _P, _I, _F, _L, _P]),
    "ds_mix_stereo": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _F, _P, _L, _P, _L, _P]),
    "ds_fftconvolve_workspace": (_I, [_P, _I, _P, _I, _P, _P, _P, _F, _P]),
    "ds_fftconvolve": (_I, [_P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _I, _F, _P, _L, _P]),
    "ds_resample_workspace": (_I, [_P, _P, _P, _P, _I, _P]),
    "ds_resample": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _P, _L, _P]),
    "ds_mask_zoom_workspace": (_I, [_P, _P, _I, _P]),
    "ds_mask_zoom": (_I, [_P, _P, _P, _P, _I, _P, _L, _P]),
    "ds_morph_rows_workspace": (_I, [_I, _I, _L, _L, _I, _P]),
    "ds_morph_rows": (_I, [_P, _P, _P, _P, _I, _I, _L, _L, _I, _P, _P, _P, _L, _P]),
    "ds_spec_images": (_I, [_P, _P, _P, _P, _I, _I, _P]),
    "ds_latent_image": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "ds_text_embed_ln": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P]),
    "ds_layernorm_rows": (_I, [_P, _P, _P, _I, _I, _F, _P]),
    "ds_text_attention": (_I, [_P, _P, _P, _I, _I, _I, _F, _P]),
    "ds_cls_gather": (_I, [_P, _P, _I, _I, _I, _P]),
    "ds_l2_normalize_rows": (_I, [_P, _I, _I, _P]),
    "ds_add_layernorm_rows_f32": (_I, [_P, _P, _P, _P, _I, _I, _F, _P]),
    # module-level entry points (csrc/engine.cu, csrc/comm.cu; structures in diffusynth_b200/engine.py)
    "ds_unet_create": (_I, [_P, _P]),
    "ds_unet_destroy": (None, [_P]),
    "ds_unet_load": (_I, [_P, C.c_char_p, _P, _P, _I]),
    "ds_unet_finalize": (_I, [_P]),
    "ds_unet_forward": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "ds_unet_plan_get": (_I, [_P, _I, _I, _I, _I, _I, _P]),
    "ds_unet_plan_run_cond": (_I, [_P, _I, _P]),
    "ds_unet_plan_run": (_I, [_P, _I, _P, _P, _P]),
    "ds_vqgan_create": (_I, [_P, _P]),
    "ds_vqgan_destroy": (None, [_P]),
    "ds_vqgan_load": (_I, [_P, C.c_char_p, _P, _P, _I]),
    "ds_vqgan_finalize": (_I, [_P]),
    "ds_vqgan_quantize": (_I, [_P, _P, _P, _P, _I, _L, _P]),
    "ds_vqgan_decode": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "ds_vqgan_encode": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "ds_sample_graph_build": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "ds_sample_graph_run": (_I, [_P, _P]),
    "ds_sample_graph_launches": (_I, [_P]),
    "ds_sample_graph_destroy": (None, [_P]),
    "ds_comm_unique_id": (_I, [_P]),
    "ds_comm_init": (_I, [_I, _I, _P, _P]),
    "ds_allgather": (_I, [_P, _P, _P, _L, _I, _P]),
    "ds_comm_destroy": (None, [_P]),
}

_lib: Optional[C.CDLL] = None


def header_symbols() -> list:
    """Every function name declared in include/diffusynth_b200.h."""
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(ds_[a-z0-9_]+)\s*\(", txt)))


def load(build: bool = True) -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if build and not os.environ.get("DS_LIB_PATH"):
        try:
            from . import _build
            if os.path.exists(_build.NVCC):
                _build.build()
        except Exception as e:  # a stale-but-present library is still usable; a missing one is fatal below
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"diffusynth_b200: building the CUDA extension failed: {e}") from e
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"diffusynth_b200: {LIB_PATH} is missing (run `python -m diffusynth_b200._build`); "
                           "there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        if os.environ.get("DS_LIB_PATH") and not hasattr(lib, name):
            continue                # A/B runs against an older build may lack newer entry points
        fn = getattr(lib, name)     # AttributeError here = header/library mismatch: fail loudly
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


class DsError(RuntimeError):
    pass


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().ds_last_error()
        raise DsError(f"{what or 'diffusynth_b200'} failed (rc={rc}): {msg.decode() if msg else ''}")
