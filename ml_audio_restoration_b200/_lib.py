"""ctypes binding of libaudiorestore_sm100.so (C-ABI in include/audiorestore.h).

There is deliberately no fallback: if the shared library has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C ml_audio_restoration_b200/csrc`)
importing the native path raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# AR_LIB_PATH: load another build of the same library (A/B measurements of kernel variants on one GPU box)
LIB_PATH = os.environ.get("AR_LIB_PATH") or os.path.join(_HERE, "libaudiorestore_sm100.so")

AR_OK, AR_ERR_INVALID, AR_ERR_WEIGHTS, AR_ERR_CUDA, AR_ERR_WORKSPACE = 0, 1, 2, 3, 4
MODEL_DENOISER, MODEL_SUPER_RES, MODEL_STEREO = 0, 1, 2
ENGINE_UMMA, ENGINE_SIMT = 0, 1
NORMALIZE_SCRATCH_BYTES = 16384
AUDIT_MAX_LAYERS = 64
HALF_MAX = 65504.0
PROFILE_CATEGORIES = ("conv", "lstm", "stem", "tail", "normalize", "chunk")


class ArTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int), ("shape", C.c_int64 * 4)]


_SIGNATURES = {
    "ar_last_error": (C.c_char_p, []),
    "ar_version": (C.c_int, []),
    "ar_set_conv_engine": (C.c_int, [C.c_int]),
    "ar_set_fusion": (C.c_int, [C.c_int]),
    "ar_model_create": (C.c_int, [C.c_int, C.POINTER(ArTensor), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "ar_model_destroy": (None, [C.c_void_p]),
    "ar_model_kind": (C.c_int, [C.c_void_p]),
    "ar_model_audit_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "ar_model_audit_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)]),
    "ar_model_audit_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "ar_model_audit_tap": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "ar_model_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "ar_model_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_stereo_forward_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_stereo_forward_window": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_chain_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ar_chain_destroy": (None, [C.c_void_p]),
    "ar_chain_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "ar_chain_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_normalize": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]),
    "ar_resample_length": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "ar_resample_mono": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "ar_pcm16_to_float": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "ar_pcm_to_float": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "ar_flac_workspace_bytes": (C.c_int, [C.c_int64, C.POINTER(C.c_size_t)]),
    "ar_flac_decode": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                 C.c_int64, C.POINTER(C.c_int64), C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_flac_encode_workspace_bytes": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_size_t),
                                                 C.POINTER(C.c_size_t)]),
    "ar_flac_encode": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                 C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p, C.c_size_t,
                                 C.c_void_p]),
    "ar_butter": (C.c_int, [C.c_int, C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ar_vinyl_mix": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int64,
                               C.c_void_p]),
    "ar_vinyl_sum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ar_filtfilt_workspace_bytes": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_size_t)]),
    "ar_filtfilt": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64,
                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ar_num_chunks": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "ar_split_chunks": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ar_overlap_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "ar_profile_enable": (C.c_int, [C.c_int]),
    "ar_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]),
    "ar_launch_count": (C.c_longlong, []),
    "ar_debug_chain_trace": (C.c_int, [C.c_void_p]),
    "ar_debug_conv1d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """Load (once) and return the native library; raise if it is not built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: the CUDA extension must be built "
                        "(__graft_entry__.build()); there is no CPU fallback")
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in _SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def check(rc: int) -> None:
    """Turn a non-zero return code into the exception the reference would raise."""
    if rc == AR_OK:
        return
    msg = (lib().ar_last_error() or b"").decode("utf-8", "replace")
    if rc == AR_ERR_INVALID and ("overlap" in msg or "empty audio" in msg or "padlen" in msg or "0 < Wn < 1" in msg):
        raise ValueError(msg)
    raise RuntimeError(msg or f"libaudiorestore error {rc}")
