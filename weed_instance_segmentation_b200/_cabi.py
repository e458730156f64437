"""ctypes binding of ``include/msda_b200.h`` (the drop-in C ABI).

The library is mandatory: using any compute entry point without
``libmsda_b200.so`` raises. There is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes
import os

import torch

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libmsda_b200.so")

ABI_VERSION = 14
MAX_LEVELS = 8
F32, BF16, U8 = 0, 1, 2
FLAG_PROFILE = 1
FLAG_BWD_V1 = 4
FLAG_STRICT_PADDING = 16
FLAG_DETERMINISTIC = 64
# retired bits (the library rejects 2 and 32): zero-valued names that bench.py still reads, so they select nothing
FLAG_BF16_ATOMICS = 0
FLAG_BWD_V2 = 0
PROF_FWD, PROF_BWD_ZERO, PROF_BWD_MAIN, PROF_BWD_CONVERT = 0, 1, 2, 3
DTYPE_CODE = {torch.float32: F32, torch.bfloat16: BF16}  # torch dtype -> the library's code (point sampling adds U8)


def ptr(t):
    """The tensor's address, or None (NULL) for a missing or empty tensor."""
    return t.data_ptr() if t is not None and t.numel() else None


class Desc(ctypes.Structure):
    """``msda_b200_desc``."""

    _fields_ = [
        ("B", ctypes.c_int32), ("S", ctypes.c_int32), ("Q", ctypes.c_int32), ("H", ctypes.c_int32),
        ("D", ctypes.c_int32), ("L", ctypes.c_int32), ("P", ctypes.c_int32),
        ("value_dtype", ctypes.c_int32), ("attn_dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
        ("spatial_shapes_hw", ctypes.POINTER(ctypes.c_int32)),
        ("level_start_index", ctypes.POINTER(ctypes.c_int64)),
    ]


_vp, _i32, _i64, _size = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
_int, _f32, _f64 = ctypes.c_int, ctypes.c_float, ctypes.c_double
_desc = ctypes.POINTER(Desc)

# name -> (restype, argtypes) of every function include/msda_b200.h declares (tests/test_abi_signatures.py checks
# each entry against the header's prototype)
SIGNATURES = {
    "msda_b200_abi_version": (_int, []),
    "msda_b200_last_error": (ctypes.c_char_p, []),
    "msda_b200_forward": (_int, [_desc, _vp, _vp, _vp, _vp, _vp, _vp]),
    "msda_b200_backward_workspace_bytes": (_size, [_desc]),
    "msda_b200_backward": (_int, [_desc, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _size, _vp, _vp]),
    "msda_b200_forward_fused": (_int, [_desc, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "msda_b200_backward_fused": (_int, [_desc, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _size, _vp, _vp]),
    "msda_b200_add_layernorm_forward": (_int, [_vp, _int, _vp, _int, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _i64, _i32,
                                               _vp]),
    "msda_b200_add_layernorm_backward": (_int, [_vp, _vp, _vp, _int, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64,
                                                _i32, _vp]),
    "msda_b200_add_layernorm_clamp_forward": (_int, [_vp, _int, _vp, _int, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp,
                                                     _i64, _i32, _vp]),
    "msda_b200_add_layernorm_clamp_backward": (_int, [_vp, _vp, _vp, _int, _vp, _int, _vp, _vp, _f32, _vp, _vp, _vp,
                                                      _vp, _vp, _vp, _i64, _i32, _vp]),
    "msda_b200_query_value_cast_forward": (_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "msda_b200_query_value_cast_backward": (_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "msda_b200_relu_backward_column_sum": (_int, [_vp, _vp, _int, _vp, _vp, _i64, _i32, _vp]),
    "msda_b200_linear_f32_available": (_int, []),
    "msda_b200_linear_f32_forward": (_int, [_vp, _vp, _vp, _int, _vp, _i64, _i32, _i32, _vp, _size, _vp]),
    "msda_b200_linear_f32_grad_input": (_int, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _size, _vp]),
    "msda_b200_linear_f32_grad_weight": (_int, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _size, _vp]),
    "msda_b200_column_sum": (_int, [_vp, _int, _vp, _i64, _i32, _vp]),
    "msda_b200_groupnorm_to_rows_forward": (_int, [_vp, _int, _vp, _vp, _f32, _vp, _i64, _vp, _i64, _i32, _i64, _i32,
                                                   _vp]),
    "msda_b200_groupnorm_to_rows_backward": (_int, [_vp, _i64, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32,
                                                    _i64, _i32, _vp]),
    "msda_b200_point_sample_forward": (_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "msda_b200_point_sample_backward": (_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "msda_b200_point_sample_backward_det_workspace_bytes": (_size, [_i64, _i32, _i64]),
    "msda_b200_point_sample_backward_det": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _i32, _vp, _size, _vp]),
    "msda_b200_resize_bilinear_backward": (_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp]),
    "msda_b200_postprocess_workspace_bytes": (_size, [_i32, _i32, _i32]),
    "msda_b200_postprocess_scores": (_int, [_vp, _i32, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _size, _vp]),
    "msda_b200_postprocess_paint": (_int, [_vp, _size, _vp, _vp, _f64, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "msda_b200_postprocess_binary_maps": (_int, [_vp, _size, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "msda_b200_host_pipeline_create": (_int, [_desc, _i32, _i32, _i32, _vp, ctypes.POINTER(_vp)]),
    "msda_b200_host_pipeline_step": (_int, [_vp] * 10),
    "msda_b200_host_pipeline_join": (_int, [_vp, _vp]),
    "msda_b200_host_pipeline_sync": (_int, [_vp]),
    "msda_b200_host_pipeline_destroy": (_int, [_vp]),
    "msda_b200_profile_ms": (_int, [_int, ctypes.POINTER(_f32)]),
    "msda_b200_launch_count": (_i64, [_int]),
}
EXPORTS = tuple(SIGNATURES)


class MSDAError(RuntimeError):
    """A non-zero return code from the C ABI."""

    def __init__(self, code: int, message: str):
        super().__init__(f"msda_b200 error {code}: {message}")
        self.code = code


_lib = None


def load() -> ctypes.CDLL:
    """Load ``libmsda_b200.so`` (building nothing; see ``build.py``). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing. Build it with `python -m weed_instance_segmentation_b200.build` "
            "(needs nvcc). This package has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    got = lib.msda_b200_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {got}, expected {ABI_VERSION}; rebuild the library")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise MSDAError(rc, load().msda_b200_last_error().decode())


_desc_cache: dict = {}


def make_desc(B, S, Q, H, D, L, P, value_dtype, attn_dtype, shapes_hw, level_start, flags=0):
    """Build a ``Desc`` plus the host arrays it points to (keep the returned tuple alive).

    Descriptors are immutable once built and the library only reads them during the call, so identical
    problems share one cached instance (saves ~9 us of ctypes marshalling per call).
    """
    key = (B, S, Q, H, D, L, P, value_dtype, attn_dtype, flags, tuple(tuple(hw) for hw in shapes_hw), tuple(level_start))
    hit = _desc_cache.get(key)
    if hit is not None:
        d, keep = hit
        d = Desc.from_buffer_copy(d)  # a private copy: callers may tweak fields (tests do)
    else:
        shp = (ctypes.c_int32 * (2 * L))(*[int(v) for hw in shapes_hw for v in hw])
        lsi = (ctypes.c_int64 * L)(*[int(v) for v in level_start])
        d0 = Desc(B, S, Q, H, D, L, P, value_dtype, attn_dtype, flags, shp, lsi)
        if len(_desc_cache) > 256:
            _desc_cache.clear()
        keep = (shp, lsi)
        _desc_cache[key] = (d0, keep)
        d = Desc.from_buffer_copy(d0)
    return d, keep


def profile_ms(which: int) -> float:
    ms = ctypes.c_float(0.0)
    check(load().msda_b200_profile_ms(which, ctypes.byref(ms)))
    return float(ms.value)


def launch_count(reset: bool = False) -> int:
    return int(load().msda_b200_launch_count(1 if reset else 0))
