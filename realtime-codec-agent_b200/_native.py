"""ctypes binding of libmagicodec_b200.so (the C ABI declared in include/magicodec_b200.h).

Only raw pointers and sizes cross the boundary; torch supplies device memory and the stream.
There is no fallback: if the library is missing or the device is not sm_100, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from .build import LIB_PATH

MC_MAX_CONVS = 8


class McSpec(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int32),
        ("n_convs", C.c_int32),
        ("conv_channels", C.c_int32 * MC_MAX_CONVS),
        ("conv_strides", C.c_int32 * MC_MAX_CONVS),
        ("d_model", C.c_int32), ("n_heads", C.c_int32), ("ffn_dim", C.c_int32),
        ("enc_layers", C.c_int32), ("dec_layers", C.c_int32),
        ("window_left", C.c_int32), ("window_right", C.c_int32),
        ("norm_eps", C.c_float),
        ("codebook_size", C.c_int32), ("codebook_dim", C.c_int32),
        ("max_positions", C.c_int32),
    ]


#: every symbol include/magicodec_b200.h declares -> (restype, argtypes)
_P, _I32, _I64 = C.c_void_p, C.c_int32, C.c_int64
SYMBOLS = {
    "mc_version": (C.c_int, []),
    "mc_last_error": (C.c_char_p, [_P]),
    "mc_create": (C.c_int, [C.POINTER(McSpec), C.c_int, C.POINTER(_P)]),
    "mc_destroy": (C.c_int, [_P]),
    "mc_set_tensor": (C.c_int, [_P, C.c_char_p, _P, _I64]),
    "mc_finalize": (C.c_int, [_P]),
    "mc_encode": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P]),
    "mc_decode": (C.c_int, [_P, _P, _I32, _I32, _I32, _P, _P]),
    "mc_decode_latents": (C.c_int, [_P, _P, _I32, _I32, _I32, _P, _P]),
    "mc_vq_search": (C.c_int, [_P, _P, _I32, _P, _P, _P]),
    "mc_codebook": (C.c_int, [_P, _P, _P]),
    "mc_launch_count": (_I64, [_P]),
    "mc_debug_trace": (_I64, [_P, _P, _I64]),
    "mc_set_debug_impl": (C.c_int, [_P, _I32, _I32]),
    "mc_set_option": (C.c_int, [_P, C.c_char_p, _I32]),
    "mc_profile_begin": (C.c_int, [_P]),
    "mc_profile_end": (C.c_int, [_P, _P, _P, _P, _P, _I32]),
    "mc_stream_create": (C.c_int, [_P, _I32, _I32, _I32, C.POINTER(_P)]),
    "mc_stream_destroy": (C.c_int, [_P]),
    "mc_stream_reset": (C.c_int, [_P]),
    "mc_stream_reset_part": (C.c_int, [_P, _I32, _I32]),
    "mc_stream_load_audio": (C.c_int, [_P, _P, _I32]),
    "mc_stream_load_codes": (C.c_int, [_P, _P, _I32]),
    "mc_stream_push_audio": (C.c_int, [_P, _P, _I32, _I32, _P, C.POINTER(_I32), _P]),
    "mc_stream_push_codes": (C.c_int, [_P, _P, _I32, _I32, _P, C.POINTER(_I32), _P]),
    "mc_stream_set_graphs": (C.c_int, [_P, _I32]),
    "mc_stream_set_emit": (C.c_int, [_P, _I32, _I32, C.c_float, C.c_float, _P]),
    "mc_stream_push_codes_emit": (C.c_int, [_P, _P, _I32, _P, C.POINTER(_I32), _P]),
    "mc_pool_create": (C.c_int, [_P, _I32, _I32, _I32, _I32, C.POINTER(_P)]),
    "mc_pool_destroy": (C.c_int, [_P]),
    "mc_pool_reset": (C.c_int, [_P, _I32, _I32, _I32]),
    "mc_pool_context_len": (C.c_int, [_P, _I32, C.POINTER(_I32), C.POINTER(_I32)]),
    "mc_pool_set_graphs": (C.c_int, [_P, _I32]),
    "mc_pool_push_audio": (C.c_int, [_P, _P, _I32, _P, _I32, _I32, _P, C.POINTER(_I32), _P]),
    "mc_pool_push_codes": (C.c_int, [_P, _P, _I32, _P, _I32, _I32, _P, C.POINTER(_I32), _P]),
    "mc_pool_set_emit": (C.c_int, [_P, _I32, _I32, C.c_float, C.c_float, _P]),
    "mc_pool_push_codes_emit": (C.c_int, [_P, _P, _I32, _P, _I32, _P, C.POINTER(_I32), _P]),
    "mc_pool_push_audio_ragged": (C.c_int, [_P, _P, _I32, _P, _I32, _I32, _P, _P]),
    "mc_pool_push_codes_ragged": (C.c_int, [_P, _P, _I32, _P, _I32, _I32, _P, _P, _P]),
    "mc_pool_push_codes_emit_ragged": (C.c_int, [_P, _P, _I32, _P, _I32, _P, _P, _P]),
    "mc_pool_graph_count": (C.c_int, [_P, C.POINTER(_I32), C.POINTER(_I32)]),
    "mc_embed_distance": (C.c_int, [_P, _P, _I32, _I32, _I64, _P, _P, _P, _P]),
    "mc_op_gemm": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _I32, _I32, _I32, _I32, _I32, _P, _I64,
                             _I32, _I32, _I64, _I64, _I32, _I32, _I32, _P]),
    "mc_op_emit_chunk": (C.c_int, [_P, _P, _I32, _I32, _I32, _I32, C.c_float, C.c_float, _P, _P, _P, _P]),
    "mc_op_embed_distance": (C.c_int, [_P, _P, _I32, _P, _I32, _I32, _I64, _P, _P, _P, _P]),
    "mc_op_pcm_to_f32": (C.c_int, [_P, _P, _I32, _I32, _I32, _I64, _I32, _P, _I64, _P]),
    "mc_op_resample": (C.c_int, [_P, _P, _I64, _I32, _I64, _I32, _I32, _P, _I32, _I64, _P, _I64, _I64, _P]),
    "mc_render_chunks": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _I32, C.c_float, C.c_float, _P, _P, _P]),
    "mc_op_f32_to_pcm": (C.c_int, [_P, _P, _I64, _I32, _I64, _I32, _P, _P]),
    "mc_flac_info": (C.c_int, [_P, _I64, C.POINTER(_I32), C.POINTER(_I32), C.POINTER(_I32), C.POINTER(_I64)]),
    "mc_flac_decode": (C.c_int, [_P, _I64, _P, _I64, C.POINTER(_I64)]),
    "mc_op_gemm_fused": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _P, _P, _I32, _P, _P, _P, _I32, _I32, _I32, _P]),
    "mc_op_rowstats": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _P]),
    "mc_op_rmsnorm": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _P]),
    "mc_op_attention": (C.c_int, [_P, _P, _P, _I32, _I32, _I32, _I32, _I32, _P]),
}

_lib: Optional[C.CDLL] = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """dlopen the engine and bind every declared symbol (raises if one is missing)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("MAGICODEC_B200_LIB") or LIB_PATH     # the env override is for diagnostic builds (build.py --trace)
    if not os.path.isfile(path):
        raise RuntimeError(
            f"{path} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc); the B200 engine has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)           # AttributeError if the .so lacks a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.mc_version() != 100:
        raise RuntimeError(f"libmagicodec_b200.so version {lib.mc_version()} != header version 100")
    _lib = lib
    return lib


class McError(RuntimeError):
    pass


def check(lib: C.CDLL, handle, rc: int, what: str) -> None:
    if rc != 0:
        msg = lib.mc_last_error(handle)
        raise McError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def current_stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream
