"""ctypes binding of lib/libtaxi2_b200.so (the C ABI in include/taxi2_b200.h).

There is no CPU fallback: importing this module without the built library, or creating an
engine without a CUDA device, raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

_PKG = Path(__file__).resolve().parent
# TAXI2_B200_LIB points at an alternative build of the same library (kernel experiments)
LIB_PATH = Path(os.environ.get("TAXI2_B200_LIB") or (_PKG / "lib" / "libtaxi2_b200.so"))

OUT_SCORE, OUT_COUNTS, OUT_METRICS = 1, 2, 4

E_ARG, E_EMPTY, E_NOMEM, E_CUDA, E_RANGE = -1, -2, -3, -4, -5


class TaxiNativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"taxi2_b200 native error {code}: {message}")
        self.code = code


_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_f64p = C.POINTER(C.c_double)
_ctx = C.c_void_p

# name -> (restype, argtypes); mirrors include/taxi2_b200.h one to one
SIGNATURES = {
    "taxi_last_error": (C.c_char_p, []),
    "taxi_abi_version": (C.c_int, []),
    "taxi_device_count": (C.c_int, []),
    "taxi_ctx_create": (C.c_int, [C.c_int, C.POINTER(_ctx)]),
    "taxi_ctx_destroy": (None, [_ctx]),
    "taxi_set_scores": (C.c_int, [_ctx, _i32p]),
    "taxi_load_sequences": (C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_int32]),
    "taxi_align_pairs": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_align_rect": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_align_rect_device": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_sync": (C.c_int, [_ctx]),
    "taxi_align_rect_both_device": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_align_rect_both": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "taxi_last_redo": (C.c_int64, [_ctx]),
    "taxi_alignment_capacity": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "taxi_align_strings": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_align_strings_metrics": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_count_rect": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "taxi_count_rect_device": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "taxi_count_pairs": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p]),
    "taxi_metrics_from_counts": (C.c_int, [_ctx, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "taxi_argmin_rows_device": (C.c_int, [_ctx, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "taxi_best_rows": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_best_rows_k": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_pairs_within": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                    C.c_int32, C.c_void_p, _i64p]),
    "taxi_pairs_within_fetch": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_clusters_within": (C.c_int, [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                       C.c_double, C.c_void_p, C.c_void_p]),
    "taxi_format_pairs": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_double,
                                    C.c_char_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "taxi_format_matrix": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_int32, C.c_double, C.c_char_p, C.c_char_p, C.c_int32]),
    "taxi_format_aligned_pairs": (C.c_int, [C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                            C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "taxi_format_values": (C.c_int64, [C.c_void_p, C.c_int64, C.c_void_p, C.c_double, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "taxi_aggregate_subsets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_void_p,
                                         C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "taxi_format_subset_rows": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                          C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int32]),
    "taxi_format_subset_matrix": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int32]),
    "taxi_host_alloc": (C.c_void_p, [C.c_int64]),
    "taxi_host_free": (None, [C.c_void_p]),
    "taxi_set_option": (C.c_int, [_ctx, C.c_char_p, C.c_int]),
    "taxi_last_kernel": (C.c_int, [_ctx]),
    "taxi_last_stats": (C.c_int, [_ctx, _i64p, _i64p, _f64p]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C taxi2_b200/csrc`. taxi2_b200 has no CPU fallback."
            )
        lib = C.CDLL(str(LIB_PATH))
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header and library out of sync
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().taxi_last_error()
        text = msg.decode("utf-8", "replace") if msg else ""
        if rc == E_EMPTY:
            raise ValueError(text or "sequence has zero length")
        raise TaxiNativeError(rc, text)
