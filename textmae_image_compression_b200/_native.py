"""ctypes binding of libtmae_b200.so (the C ABI declared in include/tmae.h).

There is no Python / CPU fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libtmae_b200.so"

TMAE_OK, TMAE_EINVAL, TMAE_ECUDA, TMAE_ESTATE, TMAE_ENOMEM = 0, 1, 2, 3, 4
FLAG_SKIP_DEAD_LRP = 1
FLAG_DEBUG_SIMT = 2
FLAG_SHARE_SM = 4
FLAG_PRECISE_RATE = 8
FLAG_PRECISE_ALL = 16
FLAG_PRECISE_X6 = 32
MODEL_GAUSSIAN, MODEL_BOTTLENECK = 0, 1
RANS_OVERRUN, RANS_UNFINISHED, RANS_BAD_INDEX, RANS_RANGE, RANS_OVERFLOW, RANS_MALFORMED = 1, 2, 4, 8, 16, 32
IMG_HEADER, IMG_CONFIG, IMG_MODEL, IMG_IDS = 64, 128, 256, 512
PIC_HEADER = 1024


class TmaeConfig(C.Structure):
    _fields_ = [
        ("img_size", C.c_int32), ("patch_size", C.c_int32), ("in_chans", C.c_int32),
        ("encoder_embed_dim", C.c_int32), ("encoder_depth", C.c_int32), ("encoder_num_heads", C.c_int32),
        ("decoder_embed_dim", C.c_int32), ("mlp_ratio", C.c_float), ("latent_depth", C.c_int32),
        ("hyperprior_depth", C.c_int32), ("num_slices", C.c_int32), ("num_keep_patches", C.c_int32),
        ("ln_eps", C.c_float), ("softmax_isa", C.c_int32), ("flags", C.c_int32),
    ]


OUTPUT_FIELDS = ("y_likelihoods", "z_likelihoods", "y_symbols", "z_symbols", "y_hat", "z_hat", "y", "z", "mu",
                 "sigma", "x_remain", "bpp", "rate_sums", "ids_shuffle", "ids_restore", "ids_keep", "y_symbols_i16",
                 "z_symbols_i16", "y_indexes")

HOST_OUTPUT_FIELDS = ("bpp", "rate_sums", "y_likelihoods", "z_likelihoods", "y_symbols", "z_symbols", "ids_restore")


class TmaeOutputs(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in OUTPUT_FIELDS]


class TmaeHostOutputs(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in HOST_OUTPUT_FIELDS]


class TmaeScoreOutputs(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in ("scores", "s_map", "t_map", "segmented")]


class TmaeProfileEntry(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_int32), ("ms", C.c_float), ("flops", C.c_double),
                ("bytes", C.c_double), ("mma_flops", C.c_double)]


class TmaeProfileStep(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("ms", C.c_float), ("flops", C.c_double), ("ctas", C.c_int32),
                ("block_n", C.c_int32)]


# every symbol include/tmae.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "tmae_abi_version": (C.c_int, []),
    "tmae_create": (C.c_int, [C.POINTER(TmaeConfig), C.POINTER(_P)]),
    "tmae_destroy": (None, [_P]),
    "tmae_last_error": (C.c_char_p, [_P]),
    "tmae_set_weight": (C.c_int, [_P, C.c_char_p, _P, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "tmae_finalize_weights": (C.c_int, [_P]),
    "tmae_enable_synthesis": (C.c_int, [_P, C.c_int, C.c_int]),
    "tmae_synthesize": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "tmae_workspace_bytes": (C.c_size_t, [_P, C.c_int]),
    "tmae_reserve": (C.c_int, [_P, C.c_int]),
    "tmae_forward": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(TmaeOutputs), _P]),
    "tmae_forward_host": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(TmaeHostOutputs), C.POINTER(TmaeOutputs), _P]),
    "tmae_set_scale_table": (C.c_int, [_P, _P, C.c_int]),
    "tmae_pack_nchw_i32": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_forward_from_latent": (C.c_int, [_P, _P, C.c_int, C.POINTER(TmaeOutputs), _P]),
    "tmae_forward_from_latent_forced": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(TmaeOutputs), _P]),
    "tmae_forward_encoder": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(TmaeOutputs), _P]),
    "tmae_decode_groups": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int]),
    "tmae_decode_begin": (C.c_int, [_P, _P, C.c_int, C.POINTER(TmaeOutputs), _P]),
    "tmae_decode_step": (C.c_int, [_P, C.c_int, _P, C.POINTER(TmaeOutputs), _P]),
    "tmae_pmf_to_quantized_cdf": (C.c_int, [_P, C.c_int, _P]),
    "tmae_rans_bound": (C.c_int64, [C.c_int64]),
    "tmae_set_cdf_tables": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "tmae_rans_encode": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "tmae_rans_decode": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, _P, C.c_int, _P, _P, _P]),
    "tmae_decompress_streams": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.POINTER(TmaeOutputs), _P, _P]),
    "tmae_rans_bound_lanes": (C.c_int64, [C.c_int64, C.c_int]),
    "tmae_rans_encode_lanes": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "tmae_rans_decode_lanes": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, _P, C.c_int, C.c_int, _P, _P, _P]),
    "tmae_decompress_streams_lanes": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, C.c_int, C.c_int, C.POINTER(TmaeOutputs), _P, _P]),
    "tmae_model_tag": (C.c_int, [_P, C.POINTER(C.c_uint32)]),
    "tmae_images_bound": (C.c_int64, [_P, C.c_int, C.c_int, C.c_int]),
    "tmae_compress_images": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "tmae_decompress_images": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, C.c_int, C.c_int, C.POINTER(TmaeOutputs), _P, _P, _P, _P]),
    "tmae_picture_tiles": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "tmae_picture_untile": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "tmae_picture_geometry": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                        C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tmae_pictures_bound": (C.c_int64, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "tmae_compress_pictures": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "tmae_decompress_pictures": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.POINTER(TmaeOutputs), _P, _P, _P, _P]),
    "tmae_mask_select": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "tmae_gaussian_rate": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "tmae_bottleneck_rate": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P]),
    "tmae_scores_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "tmae_generate_scores": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(TmaeScoreOutputs), _P, C.c_size_t, _P]),
    "tmae_huffman_create": (C.c_int, [C.POINTER(_P)]),
    "tmae_huffman_destroy": (None, [_P]),
    "tmae_huffman_last_error": (C.c_char_p, [_P]),
    "tmae_huffman_compress": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "tmae_huffman_bits": (C.c_int, [_P, _P, C.c_int64, C.c_int]),
    "tmae_huffman_code": (C.c_int, [_P, C.c_int64, C.c_char_p, C.c_int]),
    "tmae_huffman_num_symbols": (C.c_int, [_P, _P, C.c_int64]),
    "tmae_huffman_decompress": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "tmae_gemm_bf16": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_gemm_bf16_out": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_conv3x3_bf16": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_attention_bf16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_attention_hd32_bf16": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_gemm_bf16_resid": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_gemm_split": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_conv3x3_split": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "tmae_profile_enable": (C.c_int, [_P, C.c_int]),
    "tmae_profile_read": (C.c_int, [_P, C.POINTER(TmaeProfileEntry), C.c_int, C.POINTER(C.c_int)]),
    "tmae_profile_read_steps": (C.c_int, [_P, C.POINTER(TmaeProfileStep), C.c_int, C.POINTER(C.c_int)]),
    "tmae_launch_count": (C.c_int, [_P, C.c_int]),
    "tmae_attention_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "tmae_gemm_launch_plan": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tmae_conv_geometry": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int)]),
}

_lib = None


def load() -> C.CDLL:
    """Load the in-tree shared library; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            try:                                      # same image on the GPU box: nvcc is there, build in-tree
                from . import build as _build
                _build.build()
            except Exception as e:                    # noqa: BLE001
                raise RuntimeError(f"{LIB_PATH} is missing and could not be built ({e}); there is no CPU fallback") from e
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m textmae_image_compression_b200.build` "
                "(there is no CPU fallback for this path)")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error(handle=None) -> str:
    msg = load().tmae_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, handle=None, invalid_exc=ValueError):
    """Map a tmae_status to the exception class the reference would raise for the same condition."""
    if rc == TMAE_OK:
        return
    msg = last_error(handle)
    if rc == TMAE_EINVAL:
        raise invalid_exc(msg)
    if rc == TMAE_ENOMEM:
        raise MemoryError(msg)
    raise RuntimeError(f"libtmae_b200 error {rc}: {msg}")
