"""ctypes binding of ``libb200fe.so`` (the C-ABI declared in ``include/b200fe.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C csrc``.  There is no CPU
fallback: if the shared object is missing, loading raises, and every device entry point returns an
error status (turned into an exception here) when it cannot run on an sm_100 GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200FE_LIB: developer hook to load an instrumented build (e.g. the FE_GEMM_TRACE pipeline-timeline build)
LIB_PATH = os.environ.get("B200FE_LIB") or os.path.join(_HERE, "lib", "libb200fe.so")

ABI_VERSION = 1

# enums of include/b200fe.h
LOG_NONE, LOG_DB, LOG_LN = 0, 1, 2
VARIANT_AUTO, VARIANT_FFT, VARIANT_DFT_GEMM = 0, 1, 2
VARIANTS = {"auto": VARIANT_AUTO, "fft": VARIANT_FFT, "dft_gemm": VARIANT_DFT_GEMM}

OK = 0
ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_WORKSPACE, ERR_ALIGNMENT, ERR_CUDA, ERR_NO_DEVICE = -1, -2, -3, -4, -5, -6


class Params(C.Structure):
    """``b200fe_params`` (include/b200fe.h)."""

    _fields_ = [
        ("abi_version", C.c_int32),
        ("n_fft", C.c_int32),
        ("win_length", C.c_int32),
        ("hop_length", C.c_int32),
        ("n_filter", C.c_int32),
        ("n_coef", C.c_int32),
        ("log_mode", C.c_int32),
        ("top_db", C.c_float),
        ("top_db_group", C.c_int32),
        ("deltas", C.c_int32),
        ("delta_win", C.c_int32),
        ("preemph", C.c_float),
        ("cmvn", C.c_int32),
        ("variant", C.c_int32),
    ]


class B200FEError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"b200fe status {status}: {message}")
        self.status = status


# name -> (restype, argtypes); every symbol include/b200fe.h declares
_P = C.POINTER(Params)
_SIGNATURES = {
    "b200fe_version": (C.c_int32, []),
    "b200fe_last_error_string": (C.c_char_p, []),
    "b200fe_status_string": (C.c_char_p, [C.c_int32]),
    "b200fe_has_tcgen05": (C.c_int32, []),
    "b200fe_n_frames": (C.c_int64, [_P, C.c_int64]),
    "b200fe_n_out_channels": (C.c_int64, [_P]),
    "b200fe_resolve_variant": (C.c_int32, [_P]),
    "b200fe_tables_bytes": (C.c_int64, [_P]),
    "b200fe_tables_pack": (C.c_int32, [_P, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200fe_tables_variant": (C.c_int32, [_P, C.c_void_p]),
    "b200fe_workspace_bytes": (C.c_int64, [_P, C.c_int64, C.c_int64]),
    "b200fe_workspace_bytes_ex": (C.c_int64, [_P, C.c_int64, C.c_int64, C.c_int32]),
    "b200fe_spectrogram_forward": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, _P, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200fe_features_forward": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, _P, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_fbank_energies_forward": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, _P,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_lfcc_forward": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, _P, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_mel_forward": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, _P, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_compute_deltas": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200fe_host_staging_bytes": (C.c_int64, [_P, C.c_int64, C.c_int64, C.c_int32]),
    "b200fe_features_forward_host": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, _P, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_size_t, C.c_int64, C.POINTER(C.c_void_p), C.c_int32]),
    "b200fe_host_staging_bytes_i16": (C.c_int64, [_P, C.c_int64, C.c_int64, C.c_int32]),
    "b200fe_features_forward_host_i16": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, _P, C.c_void_p, C.c_void_p,
                                                     C.c_void_p, C.c_size_t, C.c_int64, C.POINTER(C.c_void_p), C.c_int32]),
    "b200fe_workspace_bytes_ragged_i16": (C.c_int64, [_P, C.c_int64, C.c_int64]),
    "b200fe_features_forward_ragged_i16": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, _P,
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_host_staging_bytes_ragged": (C.c_int64, [_P, C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "b200fe_features_forward_host_ragged": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                                        C.c_int64, C.c_int64, _P, C.c_void_p, C.c_void_p, C.c_void_p,
                                                        C.c_size_t, C.c_int64, C.POINTER(C.c_void_p), C.c_int32]),
    "b200fe_eer_workspace_bytes": (C.c_int64, [C.c_int64]),
    "b200fe_eer_min_dcf": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200fe_last_launch_count": (C.c_int64, []),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library (once) and declare every C-ABI signature.  Raises if it is missing —
    there is deliberately no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C audio-deepfake-detection-fmsl_b200/csrc`. There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.b200fe_version() != ABI_VERSION:
        raise OSError(f"libb200fe ABI {lib.b200fe_version()} != binding {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200fe_last_error_string().decode("utf-8", "replace")


def check(status: int) -> int:
    """Turn a negative status into the exception the torch-facing modules raise."""
    if status >= 0:
        return status
    msg = last_error()
    if status in (ERR_BAD_ARG,):
        raise ValueError(f"b200fe: {msg}")
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(f"b200fe: {msg}")
    raise B200FEError(status, msg)
