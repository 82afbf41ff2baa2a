"""ctypes binding of libtame_b200.so (include/tame_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the caller gets an
exception -- the product path never routes through a CPU implementation.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TAME_LIB") or os.path.join(_HERE, "libtame_b200.so")   # TAME_LIB: A/B builds

MODE_NAIVE, MODE_GOOD, MODE_BAD = 0, 1, 2
MAX_R = 8

ERRORS = {-1: "EINVAL", -2: "ECUDA", -3: "ESTATE", -4: "EHANG", -5: "ENCCL", -6: "ENOMEM"}


class TameError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libtame_b200: {ERRORS.get(code, code)}: {msg}")
        self.code = code


class TameConfig(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("T", C.c_int32), ("r", C.c_int32), ("mode", C.c_int32),
        ("lr", C.c_double), ("Rinv", C.c_double * 4),
        ("logdet_R", C.c_double), ("logdet_Q", C.c_double), ("logdet_S0", C.c_double),
        ("Phi", C.POINTER(C.c_double)), ("Qinv", C.POINTER(C.c_double)), ("S0inv", C.POINTER(C.c_double)),
        ("device", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32), ("panel", C.c_int32),
    ]


# name -> (restype, argtypes); must list every symbol declared in include/tame_b200.h
_P = C.c_void_p
_DP = C.POINTER(C.c_double)
SIGNATURES = {
    "tame_version": (C.c_char_p, []),
    "tame_last_error": (C.c_char_p, []),
    "tame_launch_count": (C.c_int64, []),
    "tame_create": (C.c_int, [C.POINTER(TameConfig), C.POINTER(_P)]),
    "tame_destroy": (C.c_int, [_P]),
    "tame_set_stream": (C.c_int, [_P, _P]),
    "tame_local_rows": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "tame_bind_Y": (C.c_int, [_P, _P]),
    "tame_bind_Y_f32": (C.c_int, [_P, _P]),
    "tame_bind_state": (C.c_int, [_P, _P, _P]),
    "tame_sweep": (C.c_int, [_P]),
    "tame_elbo_mse": (C.c_int, [_P, _DP]),
    "tame_iterate": (C.c_int, [_P, _DP]),
    "tame_fit": (C.c_int, [_P, C.c_int32, C.c_double, _DP, _DP, C.POINTER(C.c_int32)]),
    "tame_fit_device": (C.c_int, [_P, C.c_int32, C.c_double, _P, _P, _P]),
    "tame_fit_host": (C.c_int, [C.POINTER(TameConfig), _P, _P, _P, C.c_int32, C.c_double, _DP, _DP, C.POINTER(C.c_int32)]),
    "tame_fit_host_f32": (C.c_int, [C.POINTER(TameConfig), _P, _P, _P, C.c_int32, C.c_double, _DP, _DP, C.POINTER(C.c_int32)]),
    "tame_fit_batch": (C.c_int, [C.c_int32, C.POINTER(TameConfig), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.c_int32,
                                C.c_double, _DP, _DP, C.POINTER(C.c_int32), C.c_int32]),
    "tame_fit_batch_f32": (C.c_int, [C.c_int32, C.POINTER(TameConfig), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.c_int32,
                                    C.c_double, _DP, _DP, C.POINTER(C.c_int32), C.c_int32]),
    "tame_generate_Y": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _DP, _P, C.c_uint64, C.c_int32, C.c_int32, _P, _P]),
    "tame_generate_Y_f32": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _DP, _P, C.c_uint64, C.c_int32, C.c_int32, _P, _P]),
    "tame_align_states": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P, _P, _DP, _P]),
    "tame_align_signs": (C.c_int, [C.c_int64, C.c_int32, _P, _P, _P, _DP, _P]),
    "tame_procrustes": (C.c_int, [C.c_int32, C.c_int32, _P, _P, C.c_int32, _P, _P, _P]),
    "tame_contributions": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P, _P]),
    "tame_uv_correlation": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "tame_state_mse": (C.c_int, [C.c_int64, _P, _P, _DP, _P]),
    "tame_comm_unique_id": (C.c_int, [_P]),
    "tame_comm_init": (C.c_int, [_P, _P]),
    "tame_ipc_export": (C.c_int, [_P, _P]),
    "tame_ipc_import": (C.c_int, [_P, _P]),
    "tame_peer_attach": (C.c_int, [_P, _P]),
    "tame_gather_state": (C.c_int, [_P]),
    "tame_last_timing": (C.c_int, [_P, _DP, _DP, _DP, _DP, _DP]),
    "tame_set_timing": (C.c_int, [_P, C.c_int32]),
    "tame_y_symmetric": (C.c_int, [_P]),
    "tame_debug_probes": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "tame_debug_trace": (C.c_int, [_P, C.POINTER(C.c_uint64), C.c_int32]),
}

_lib = None


def load():
    """Load libtame_b200.so; raises (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(make -C python-temporal-ame-svi_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise TameError(rc, load().tame_last_error().decode())


def dptr(arr):
    """numpy float64 C-contiguous array -> POINTER(c_double)"""
    return arr.ctypes.data_as(_DP)
