"""ctypes binding of libtts_b200.so (include/tts_b200.h).  Fails loudly when the CUDA library is
missing -- there is no CPU or PyTorch fallback on the product path."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libtts_b200.so")


class TtsConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32)] + [(n, C.c_int32) for n in (
        "n_vocab", "d_model", "n_heads", "n_enc_layers", "n_dec_layers", "d_ff", "n_mels", "d_prenet",
        "enc_conv_layers", "conv_kernel", "postnet_channels", "postnet_layers", "max_pos")] + [
        ("ln_eps", C.c_float), ("bn_eps", C.c_float)]


_P, _I, _I64, _U64, _SZ = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); every symbol include/tts_b200.h declares
SIGNATURES = {
    "tts_version": (C.c_char_p, []),
    "tts_launch_count": (C.c_ulonglong, []),
    "tts_create": (_I, [C.POINTER(TtsConfig), _I, C.POINTER(_P)]),
    "tts_destroy": (_I, [_P]),
    "tts_last_error_string": (C.c_char_p, [_P]),
    "tts_load_weight": (_I, [_P, C.c_char_p, _P, _I64]),
    "tts_finalize_weights": (_I, [_P]),
    "tts_set_option": (_I, [_P, C.c_char_p, _I64]),
    "tts_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "tts_encode": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "tts_decode_begin": (_I, [_P, _P, _I, _I, _I, _U64, _I, _P]),
    "tts_decode_steps": (_I, [_P, _P, _I, _P]),
    "tts_decode_status": (_I, [_P, _P, C.POINTER(_I), C.POINTER(_I), _P]),
    "tts_decode_end": (_I, [_P, _P, _I, _P, _P, _P, _P, _P]),
    "tts_decode_set_batch": (_I, [_P, _P, _P, _P, _I, _P]),
    "tts_decode_set_frame": (_I, [_P, _P, _I, _P, _P]),
    "tts_decode_get_frame": (_I, [_P, _P, _I, _P, _P, _P]),
    "tts_stream_scratch_bytes": (_SZ, [_P, _I, _I]),
    "tts_decode_emit": (_I, [_P, _P, _P, _SZ, _I, _I, _P, _P, _P, _P, _P]),
    "tts_infer_host": (_I, [_P, _P, _P, _P, _I, _I, _I, _U64, _I, _P, _P, _P, C.POINTER(_I), _P]),
    "tts_forward": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _U64, _I, _P, _P, _P, _P]),
    "tts_align_scratch_bytes": (_SZ, [_P, _I, _I, _I]),
    "tts_forward_align": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _U64, _I, C.c_uint32, _I] + [_P] * 8),
    "tts_debug_phase_timestamps": (_I, [_P, _P, _P, _I, _P]),
    "tts_debug_read_dump": (_I, [_P, _P, _I64, _I64, _P, _P]),
    "tts_debug_kv_index": (_I, [_I, _I, _I]),
    "tts_debug_pack_segment": (_I64, [_P, _I, _I, _P, _I, _I, _I, _I, _P, _I64]),
    "tts_train_begin": (_I, [_P]),
    "tts_train_end": (_I, [_P]),
    "tts_train_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "tts_train_step": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _U64, _I, C.c_double, C.c_float, _P, _P]),
    "tts_train_outputs": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "tts_train_grads": (_I, [_P, C.POINTER(_P), C.POINTER(_I64)]),
    "tts_train_adam": (_I, [_P, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    "tts_train_ipc_handles": (_I, [_P, _P, _P]),
    "tts_train_set_peers": (_I, [_P, _I, _I, _P, _P]),
    "tts_train_adam_peers": (_I, [_P, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    "tts_train_repack": (_I, [_P, _P]),
    "tts_train_num_tensors": (_I, [_P]),
    "tts_train_tensor_info": (_I, [_P, _I, C.POINTER(C.c_char_p), C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_I)]),
    "tts_train_read": (_I, [_P, _I, _I64, _I64, _P]),
    "tts_train_write": (_I, [_P, _I, _I64, _I64, _P]),
    "tts_train_forward": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _U64, _I, C.c_double, _P]),
    "tts_train_backward": (_I, [_P, _P, _I, _I, _I, _I, C.c_double, _P, _P, _P, _P]),
    "tts_k_gemm": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "tts_k_conv5": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "tts_k_attention": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "tts_k_attention_lse": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "tts_k_attention_bwd": (_I, [_P] * 11 + [_I, _I, _I, _I, _I, _P]),
    "tts_k_cross_align": (_I, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "tts_k_layernorm": (_I, [_P, _P, _P, _P, _I, C.c_float, _P]),
    "tts_k_philox_bits": (_I, [_U64, _I, _I, _I, _I, _I, _P, _P]),
    "tts_k_wgrad": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "tts_k_dgrad": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P, _P]),
    "tts_k_bn_train_fwd": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, C.c_float, _I, _I, _P, _I, _P, _I, _P, _P, _P, _P]),
    "tts_k_bn_train_bwd": (_I, [_P, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, C.c_float, _I, _I, _P, _I, _P, _P, _P, _I, _P]),
    "tts_k_ln_bwd": (_I, [_P, _P, _P, C.c_float, _I, _I, _P, _P, _I, _P, _I, C.c_uint32, C.c_float, _P, _P, _P]),
    "tts_k_loss": (_I, [_P, _P, _P, _P, _P, _I, _I, C.c_float, _P, _P, _P, _P, _P, _P]),
    "tts_k_head_grad": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _P, _P]),
    "tts_k_dropw_bwd": (_I, [_P, _P, _I, _I, _I, _P, _I, C.c_uint32, C.c_float, _P, _P, _I, _P]),
    "tts_k_embed_bwd": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
}

_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """dlopen the in-tree library (building it with nvcc first if it is absent or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and _build.needs_build():
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m transformer_tacotron2_b200.build` "
                           "(there is no CPU fallback for the B200 path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


class TtsError(RuntimeError):
    pass


def check(lib, handle, rc: int, what: str) -> None:
    if rc != 0:
        detail = lib.tts_last_error_string(handle).decode() if handle else ""
        kind = "argument/state error" if rc < 0 else "cudaError"
        raise TtsError(f"{what} failed: {kind} {rc} {detail}")
