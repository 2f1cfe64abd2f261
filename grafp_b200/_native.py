"""ctypes binding of libgrafp_b200.so (the C ABI declared in include/grafp_b200.h).

There is no fallback: if the library is missing, or a call fails, a RuntimeError is
raised.  Tensors are passed as raw device pointers, the stream as the current torch
CUDA stream handle.
"""
from __future__ import annotations

import ctypes
import os
import threading

from . import build as _build

_c = ctypes
_vp, _i, _sz = _c.c_void_p, _c.c_int, _c.c_size_t

# name -> (restype, argtypes); mirrors include/grafp_b200.h one to one
SIGNATURES = {
    "grafp_abi_version": (_i, []),
    "grafp_last_error": (_c.c_char_p, []),
    "grafp_set_option": (_i, [_c.c_char_p, _i]),
    "grafp_get_option": (_i, [_c.c_char_p]),
    "grafp_check_index": (_i, [_vp, _i, _c.c_longlong, _i, _vp, _vp]),
    "grafp_knn_last_algo": (_c.c_char_p, []),
    "grafp_knn_last_variant": (_c.c_char_p, []),
    "grafp_knn_workspace_bytes": (_sz, [_i] * 6),
    "grafp_knn_fwd": (_i, [_vp] * 5 + [_i] * 11 + [_vp, _sz, _vp]),
    "grafp_mr_aggregate_fwd": (_i, [_vp] * 4 + [_i] + [_vp] * 2 + [_i] * 6 + [_vp]),
    "grafp_mr_aggregate_bwd_workspace_bytes": (_sz, [_i] * 3),
    "grafp_mr_aggregate_bwd": (_i, [_vp] * 4 + [_i] + [_vp] * 2 + [_i] * 6 + [_vp, _sz, _vp]),
    "grafp_gather_fwd": (_i, [_vp] * 2 + [_i] + [_vp] + [_i] * 6 + [_vp]),
    "grafp_gather_bwd": (_i, [_vp] * 2 + [_i] + [_vp] + [_i] * 6 + [_vp]),
    "grafp_neighbor_sum_fwd": (_i, [_vp] * 2 + [_i] + [_vp] + [_i] * 6 + [_vp]),
    "grafp_neighbor_sum_bwd": (_i, [_vp] * 2 + [_i] + [_vp] + [_i] * 6 + [_vp]),
    "grafp_edge_gather_fwd": (_i, [_vp] * 4 + [_i] + [_vp] + [_i] * 6 + [_vp]),
    "grafp_edge_gather_bwd": (_i, [_vp] * 3 + [_i] + [_vp] * 2 + [_i] * 6 + [_vp]),
    "grafp_max_over_k_fwd": (_i, [_vp] * 3 + [_i] * 5 + [_vp]),
    "grafp_max_over_k_bwd": (_i, [_vp] * 3 + [_i] * 5 + [_vp]),
    "grafp_peak_extract_workspace_bytes": (_sz, [_i] * 3),
    "grafp_peak_extract_fwd": (_i, [_vp] * 4 + [_i] * 7 + [_vp]),
    "grafp_peak_extract_bwd": (_i, [_vp] * 4 + [_sz] + [_vp] * 2 + [_i] * 7 + [_vp]),
    "grafp_ntxent_fwd": (_i, [_vp] * 4 + [_i, _i, _c.c_float, _vp]),
    "grafp_ntxent_bwd": (_i, [_vp] * 4 + [_i, _i, _c.c_float, _vp]),
    "grafp_bn_workspace_bytes": (_sz, [_i]),
    "grafp_bn_train_fwd": (_i, [_vp] * 11 + [_c.c_longlong, _i, _c.c_float, _c.c_float, _i, _i, _vp, _sz, _vp]),
    "grafp_bn_train_bwd": (_i, [_vp] * 10 + [_c.c_longlong, _i, _i, _i, _vp, _sz, _vp]),
    "grafp_ntxent_rows_fwd": (_i, [_vp] * 4 + [_i, _i, _i, _i, _c.c_float, _vp]),
    "grafp_ntxent_rows_bwd": (_i, [_vp] * 4 + [_i, _i, _i, _i, _c.c_float, _c.c_float, _vp]),
    "grafp_downsample_taps_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "grafp_downsample_taps_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "grafp_conv1x1_bn_stats_supported": (_i, [_c.c_longlong, _i, _i, _i, _i]),
    "grafp_conv1x1_bn_stats_fwd": (_i, [_vp] * 3 + [_c.c_longlong, _i, _i, _i, _i, _vp, _sz, _vp]),
    "grafp_bn_train_fwd_from_moments": (_i, [_vp] * 11 + [_c.c_longlong, _i, _c.c_float, _c.c_float, _i, _i, _vp, _sz, _vp]),
    "grafp_search_prepare": (_i, [_vp, _c.c_longlong, _i, _vp, _vp, _vp, _vp]),
    "grafp_search_workspace_bytes": (_sz, [_i] * 4),
    "grafp_search_fwd": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
}

ABI_VERSION = 7
KNN_AUTO, KNN_SIMT, KNN_TC, KNN_TC_TF32 = 0, 1, 2, 3
KNN_MAX_K = 128
METRIC_L2, METRIC_COSINE = 0, 1

_lib = None
_lock = threading.Lock()


def library_path() -> str:
    return os.environ.get("GRAFP_B200_LIB", _build.LIB_PATH)


def load() -> ctypes.CDLL:
    """Load (once) and type the shared library; raises if it is absent or has the wrong ABI."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.isfile(path):
            raise RuntimeError(
                f"grafp_b200: native library {path} not found. Build it with "
                "`python -m grafp_b200.build` (needs nvcc); there is no PyTorch/CPU fallback.")
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
            fn.restype, fn.argtypes = res, args
        got = lib.grafp_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"grafp_b200: {path} has ABI version {got}, expected {ABI_VERSION}")
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().grafp_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"grafp_b200.{what} failed (code {rc}): {msg}")
