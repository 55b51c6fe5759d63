"""ctypes binding of libinfernos_b200.so (the C-ABI declared in include/infernos_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, a RuntimeError is raised
(the reference's error convention: RuntimeError out of infer(), /root/reference/Cluster/InfernTTSWorker.py:87-91).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int16, c_int32, c_int64, c_size_t, c_uint8, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("B2_SO_PATH") or os.path.join(HERE, "libinfernos_b200.so")      # B2_SO_PATH: a variant build for A/B runs

MODE_FP32, MODE_BF16 = 0, 1
LAW_ULAW, LAW_ALAW, LAW_NONE = 0, 1, -1
TAIL_APPLY_POSTNET = 1

# name -> (restype, argtypes); must list every symbol of include/infernos_b200.h (tests check that)
SIGNATURES = {
    "b2_abi_version": (c_int, []),
    "b2_last_error": (c_char_p, [c_void_p]),
    "b2_ctx_create": (c_void_p, [c_int, c_int, c_int, c_int]),
    "b2_ctx_destroy": (None, [c_void_p]),
    "b2_ctx_mode": (c_int, [c_void_p]),
    "b2_ctx_device_bytes": (c_size_t, [c_void_p]),
    "b2_load_vocoder_tensor": (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int]),
    "b2_load_chunker_tensor": (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int]),
    "b2_load_postnet_tensor": (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int]),
    "b2_weights_finalize": (c_int, [c_void_p]),
    "b2_set_resample_taps": (c_int, [c_void_p, c_void_p]),
    "b2_vocoder_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "b2_chunker_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "b2_resample_2to1": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p, c_void_p]),
    "b2_tts_tail": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2_tts_tail_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2_postnet_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "b2_tts_tail2": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2_tts_tail_host2": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2_ctx_poll_errors": (c_int, [c_void_p, c_void_p]),
    "b2_debug_set_taps": (c_int, [c_void_p, c_void_p]),
    "b2_sched_create": (c_void_p, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2_sched_destroy": (None, [c_void_p]),
    "b2_sched_set_policy": (c_int, [c_void_p, c_int, c_int]),
    "b2_sched_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "b2_sched_poll": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int]),
    "b2_sched_flush": (c_int, [c_void_p, c_int]),
    "b2_sched_get_stats": (c_int, [c_void_p, c_void_p]),
    "b2_sched_prebuild": (c_int, [c_void_p, c_int]),
    "b2_tts_server_create": (c_void_p, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float, c_float, c_uint64]),
    "b2_tts_server_destroy": (None, [c_void_p]),
    "b2_tts_server_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "b2_tts_server_cancel": (c_int, [c_void_p, c_void_p, c_int]),
    "b2_tts_server_poll": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int]),
    "b2_tts_server_flush": (c_int, [c_void_p, c_int]),
    "b2_tts_server_get_stats": (c_int, [c_void_p, c_void_p]),
    "b2_dec_create": (c_void_p, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2_dec_destroy": (None, [c_void_p]),
    "b2_dec_device_bytes": (c_size_t, [c_void_p]),
    "b2_dec_load_tensor": (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int]),
    "b2_dec_finalize": (c_int, [c_void_p]),
    "b2_dec_start": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b2_dec_steps": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_uint64, c_void_p, c_void_p, c_void_p]),
    "b2_dec_poll_errors": (c_int, [c_void_p, c_void_p]),
    "b2_dec_set_graphs": (c_int, [c_void_p, c_int]),
    "b2_dec_get_step": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "b2_enc_create": (c_void_p, [c_int, c_int, c_int, c_int]),
    "b2_enc_destroy": (None, [c_void_p]),
    "b2_enc_device_bytes": (c_size_t, [c_void_p]),
    "b2_enc_load_tensor": (c_int, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int]),
    "b2_enc_finalize": (c_int, [c_void_p]),
    "b2_enc_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "b2_enc_poll_errors": (c_int, [c_void_p, c_void_p]),
    "b2_session_reset": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "b2_session_get_pre_frames": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "b2_session_set_pre_frames": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "b2_g711_encode_f32": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_g711_encode_i16": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_f32_to_pcm16": (c_int, [c_void_p, c_size_t, c_void_p, c_void_p]),
    "b2_g711_decode_f32": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_g711_decode_i16": (c_int, [c_void_p, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_resample_g711_encode": (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_g711_decode_upsample": (c_int, [c_void_p, c_size_t, c_size_t, c_int, c_void_p, c_void_p]),
    "b2_resample_1to2": (c_int, [c_void_p, c_size_t, c_size_t, c_void_p, c_void_p]),
    "b2_g711_decode_ragged": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p, c_void_p]),
    "b2_g711_decode_many_host": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p, c_void_p]),
    "b2_conv1d_tc": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p]),
    "b2_conv1d_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p]),
    "b2_linear": (c_int, [c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                          POINTER(c_int), c_void_p]),
    "b2_resblock_tc": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_float, c_float, c_float, c_void_p]),
    "b2_resblock_t_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int)]),
    "b2_debug_set_stacked_min_taps": (c_int, [c_int]),
    "b2_kernel_launch_count": (c_uint64, []),
    "b2_profile_begin": (c_int, [c_void_p]),
    "b2_profile_end": (c_int, [c_void_p, POINTER(ctypes.c_double), POINTER(c_uint64)]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Loads the library (once).  Raises RuntimeError when it has not been built: no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -m infernos_b200.build` (nvcc, sm_100a). "
            "infernos_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.b2_abi_version() != 1:
        raise RuntimeError("libinfernos_b200.so has an unexpected ABI version")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().b2_last_error(None)
        raise RuntimeError(f"infernos_b200 {what}: {msg.decode() if msg else 'error'}")
