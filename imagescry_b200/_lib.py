"""ctypes binding of libimagescry_b200.so (the C ABI in include/imagescry_b200.h).

There is no fallback: if the shared library is missing or a call fails, the caller gets an
exception.  Torch is used only to obtain device pointers, the current stream and allocations.
"""

from __future__ import annotations

import ctypes
import os
import threading
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p, POINTER

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "lib", "libimagescry_b200.so")

OK = 0
ERR_INVALID_ARG = -1
ERR_CUDA = -2
ERR_UNSUPPORTED = -3
ERR_WORKSPACE = -4

LAYOUT_NCHW = 0
LAYOUT_NHWC = 1
DTYPE_U8 = 0
DTYPE_F32 = 1
DTYPE_BF16 = 2
KNN_CONTINUE = 1
KNN_NO_FINALIZE = 2
KNN_EXCLUDE_SELF = 4
KNN_PACKED = 8
KNN_RANGE_WORKSPACE_BYTES = 2048  # ISX_KNN_RANGE_WORKSPACE_BYTES

# name -> (restype, argtypes); mirrors include/imagescry_b200.h one to one
SIGNATURES: dict[str, tuple] = {
    "isx_abi_version": (c_int, []),
    "isx_last_error": (c_char_p, []),
    "isx_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "isx_preprocess_stats_workspace_bytes": (c_size_t, [c_int]),
    "isx_preprocess_stats": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_preprocess_apply": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_float,
         c_int, c_float, c_int, c_float, c_void_p, c_int, c_void_p],
    ),
    "isx_preprocess_patches_stats": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
         c_void_p],
    ),
    "isx_preprocess_patches_apply": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_int,
         c_float, c_int, c_float, c_void_p, c_int, c_void_p],
    ),
    "isx_resize_bilinear": (
        c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    ),
    "isx_project_packed_bytes": (c_size_t, [c_int, c_int]),
    "isx_project_pack": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_int64, c_void_p, c_size_t, c_void_p]),
    "isx_l2norm_project_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "isx_l2norm_project": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_l2norm_project_fp16": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_l2norm_cells": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "isx_pca_moments_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "isx_pca_moments": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isx_row_rnorm_bf16": (c_int, [c_void_p, c_int64, c_int, c_float, c_void_p, c_void_p]),
    "isx_maps_to_rows_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p]),
    "isx_knn_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "isx_knn_search": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p,
         c_void_p, c_size_t, c_void_p],
    ),
    "isx_knn_search_ex": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int64, c_int, c_void_p,
         c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_knn_search_scatter": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int64, c_int, c_void_p, c_int,
         c_int, c_void_p, c_size_t, c_void_p],
    ),
    "isx_topk_merge": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "isx_topk_merge_packed": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "isx_knn_search_grouped": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p,
         c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_topk_merge_grouped": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "isx_knn_range": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_float, c_int64, c_int64, c_int, c_void_p,
         c_int64, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "isx_knn_range_sort_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "isx_knn_range_sort": (
        c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    ),
    "isx_quantize_rows_e4m3": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "isx_knn_search_fp8": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p,
         c_size_t, c_void_p],
    ),
    "isx_knn_rescore": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int64, c_int, c_void_p,
         c_void_p, c_void_p],
    ),
    "isx_knn_maxsim": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int64, c_int64, c_void_p, c_void_p,
         c_size_t, c_void_p],
    ),
    "isx_maxsim_sets_topk": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p],
    ),
    "isx_roi_rasterize":(c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int64, c_void_p, c_void_p]),
    "isx_masked_pool": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int64, c_void_p, c_void_p]),
}

_lock = threading.Lock()
_lib: ctypes.CDLL | None = None


class IsxError(RuntimeError):
    """A CUDA-side failure reported by the library (ISX_ERR_CUDA / ISX_ERR_WORKSPACE)."""


def load() -> ctypes.CDLL:
    """Load the shared library (once).  Raises if it has not been built — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m imagescry_b200._build` "
                "(imagescry_b200 has no CPU or PyTorch fallback)"
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.isx_abi_version() != 1:
            raise RuntimeError(f"ABI mismatch: library reports {lib.isx_abi_version()}, binding expects 1")
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    """Map a status code to the exception the reference's API would raise."""
    if rc == OK:
        return
    msg = load().isx_last_error().decode("utf-8", "replace")
    if rc in (ERR_INVALID_ARG, ERR_UNSUPPORTED):
        raise ValueError(f"{what}: {msg}")
    raise IsxError(f"{what}: {msg} (code {rc})")


def require_cuda(t, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} must be a CUDA tensor (got device {t.device}); imagescry_b200 runs on the GPU only "
            "and has no CPU fallback"
        )


def stream_ptr(device) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream


class on_device:
    """Context manager for one C-ABI call: makes the operands' device the CURRENT device (the library
    launches on the current device, reads its SM count and encodes its tensor maps there) and yields
    the pointer of that device's current stream.  Operands on different devices are rejected —
    the reference is plain torch and raises for mixed devices too."""

    def __init__(self, *tensors) -> None:
        import torch

        devs = {t.device for t in tensors if t is not None}
        if len(devs) != 1:
            raise ValueError(f"all operands of one call must live on the same CUDA device, got {sorted(map(str, devs))}")
        (self.device,) = devs
        if self.device.type != "cuda":
            raise RuntimeError(
                f"operands must be CUDA tensors (got device {self.device}); imagescry_b200 runs on the GPU only "
                "and has no CPU fallback"
            )
        self._guard = torch.cuda.device(self.device)

    def __enter__(self) -> int:
        self._guard.__enter__()
        return stream_ptr(self.device)

    def __exit__(self, *exc):
        return self._guard.__exit__(*exc)
