"""ctypes binding of ``include/msda_b200.h`` (the drop-in C ABI).

The library is mandatory: using any compute entry point without
``libmsda_b200.so`` raises. There is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes
import os

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

# every symbol include/msda_b200.h declares
EXPORTS = (
    "msda_b200_abi_version",
    "msda_b200_last_error",
    "msda_b200_forward",
    "msda_b200_backward_workspace_bytes",
    "msda_b200_backward",
    "msda_b200_forward_fused",
    "msda_b200_backward_fused",
    "msda_b200_add_layernorm_forward",
    "msda_b200_add_layernorm_backward",
    "msda_b200_add_layernorm_clamp_forward",
    "msda_b200_add_layernorm_clamp_backward",
    "msda_b200_query_value_cast_forward",
    "msda_b200_query_value_cast_backward",
    "msda_b200_relu_backward_column_sum",
    "msda_b200_linear_f32_available",
    "msda_b200_linear_f32_forward",
    "msda_b200_linear_f32_grad_input",
    "msda_b200_linear_f32_grad_weight",
    "msda_b200_column_sum",
    "msda_b200_groupnorm_to_rows_forward",
    "msda_b200_groupnorm_to_rows_backward",
    "msda_b200_point_sample_forward",
    "msda_b200_point_sample_backward",
    "msda_b200_point_sample_backward_det_workspace_bytes",
    "msda_b200_point_sample_backward_det",
    "msda_b200_resize_bilinear_backward",
    "msda_b200_host_pipeline_create",
    "msda_b200_host_pipeline_step",
    "msda_b200_host_pipeline_join",
    "msda_b200_host_pipeline_sync",
    "msda_b200_host_pipeline_destroy",
    "msda_b200_profile_ms",
    "msda_b200_launch_count",
)


class Desc(ctypes.Structure):
    """``msda_b200_desc``."""

    _fields_ = [
        ("B", ctypes.c_int32), ("S", ctypes.c_int32), ("Q", ctypes.c_int32), ("H", ctypes.c_int32),
        ("D", ctypes.c_int32), ("L", ctypes.c_int32), ("P", ctypes.c_int32),
        ("value_dtype", ctypes.c_int32), ("attn_dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
        ("spatial_shapes_hw", ctypes.POINTER(ctypes.c_int32)),
        ("level_start_index", ctypes.POINTER(ctypes.c_int64)),
    ]


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
    vp = ctypes.c_void_p
    dp = ctypes.POINTER(Desc)
    lib.msda_b200_abi_version.restype = ctypes.c_int
    lib.msda_b200_abi_version.argtypes = []
    lib.msda_b200_last_error.restype = ctypes.c_char_p
    lib.msda_b200_last_error.argtypes = []
    lib.msda_b200_forward.restype = ctypes.c_int
    lib.msda_b200_forward.argtypes = [dp, vp, vp, vp, vp, vp, vp]
    lib.msda_b200_backward_workspace_bytes.restype = ctypes.c_size_t
    lib.msda_b200_backward_workspace_bytes.argtypes = [dp]
    lib.msda_b200_backward.restype = ctypes.c_int
    lib.msda_b200_backward.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp, ctypes.c_size_t, vp, vp]
    lib.msda_b200_forward_fused.restype = ctypes.c_int
    lib.msda_b200_forward_fused.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.msda_b200_backward_fused.restype = ctypes.c_int
    lib.msda_b200_backward_fused.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ctypes.c_size_t, vp, vp]
    lib.msda_b200_add_layernorm_forward.restype = ctypes.c_int
    lib.msda_b200_add_layernorm_forward.argtypes = [vp, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_float, vp, vp, vp, vp,
                                                    ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_add_layernorm_backward.restype = ctypes.c_int
    lib.msda_b200_add_layernorm_backward.argtypes = [vp, vp, vp, ctypes.c_int, vp, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp,
                                                     ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_add_layernorm_clamp_forward.restype = ctypes.c_int
    lib.msda_b200_add_layernorm_clamp_forward.argtypes = [vp, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_float,
                                                          ctypes.c_float, vp, vp, vp, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_add_layernorm_clamp_backward.restype = ctypes.c_int
    lib.msda_b200_add_layernorm_clamp_backward.argtypes = [vp, vp, vp, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_float,
                                                           vp, vp, vp, vp, vp, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_query_value_cast_forward.restype = ctypes.c_int
    lib.msda_b200_query_value_cast_forward.argtypes = [vp, vp, vp, vp, ctypes.c_int64, vp]
    lib.msda_b200_query_value_cast_backward.restype = ctypes.c_int
    lib.msda_b200_query_value_cast_backward.argtypes = [vp, vp, vp, vp, ctypes.c_int64, vp]
    lib.msda_b200_linear_f32_available.restype = ctypes.c_int
    lib.msda_b200_linear_f32_available.argtypes = []
    lib.msda_b200_linear_f32_forward.restype = ctypes.c_int
    lib.msda_b200_linear_f32_forward.argtypes = [vp, vp, vp, ctypes.c_int, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                                 vp, ctypes.c_size_t, vp]
    for fn in (lib.msda_b200_linear_f32_grad_input, lib.msda_b200_linear_f32_grad_weight):
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, vp, ctypes.c_size_t, vp]
    lib.msda_b200_relu_backward_column_sum.restype = ctypes.c_int
    lib.msda_b200_relu_backward_column_sum.argtypes = [vp, vp, ctypes.c_int, vp, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_column_sum.restype = ctypes.c_int
    lib.msda_b200_column_sum.argtypes = [vp, ctypes.c_int, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_groupnorm_to_rows_forward.restype = ctypes.c_int
    lib.msda_b200_groupnorm_to_rows_forward.argtypes = [vp, ctypes.c_int, vp, vp, ctypes.c_float, vp, ctypes.c_int64, vp,
                                                        ctypes.c_int64, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_groupnorm_to_rows_backward.restype = ctypes.c_int
    lib.msda_b200_groupnorm_to_rows_backward.argtypes = [vp, ctypes.c_int64, vp, ctypes.c_int, vp, vp, vp, vp, vp, vp,
                                                         ctypes.c_int64, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_point_sample_forward.restype = ctypes.c_int
    lib.msda_b200_point_sample_forward.argtypes = [vp, vp, vp, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_point_sample_backward.restype = ctypes.c_int
    lib.msda_b200_point_sample_backward.argtypes = [vp, vp, vp, vp, ctypes.c_int64, ctypes.c_int32, vp]
    lib.msda_b200_point_sample_backward_det_workspace_bytes.restype = ctypes.c_size_t
    lib.msda_b200_point_sample_backward_det_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int64]
    lib.msda_b200_point_sample_backward_det.restype = ctypes.c_int
    lib.msda_b200_point_sample_backward_det.argtypes = [vp, vp, vp, ctypes.c_int64, vp, vp, ctypes.c_int64, ctypes.c_int32,
                                                        vp, ctypes.c_size_t, vp]
    lib.msda_b200_resize_bilinear_backward.restype = ctypes.c_int
    lib.msda_b200_resize_bilinear_backward.argtypes = [vp, vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                                       ctypes.c_int32, ctypes.c_int32, vp]
    lib.msda_b200_host_pipeline_create.restype = ctypes.c_int
    lib.msda_b200_host_pipeline_create.argtypes = [dp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp,
                                                   ctypes.POINTER(vp)]
    lib.msda_b200_host_pipeline_step.restype = ctypes.c_int
    lib.msda_b200_host_pipeline_step.argtypes = [vp] * 10
    lib.msda_b200_host_pipeline_join.restype = ctypes.c_int
    lib.msda_b200_host_pipeline_join.argtypes = [vp, vp]
    lib.msda_b200_host_pipeline_sync.restype = ctypes.c_int
    lib.msda_b200_host_pipeline_sync.argtypes = [vp]
    lib.msda_b200_host_pipeline_destroy.restype = ctypes.c_int
    lib.msda_b200_host_pipeline_destroy.argtypes = [vp]
    lib.msda_b200_profile_ms.restype = ctypes.c_int
    lib.msda_b200_profile_ms.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    lib.msda_b200_launch_count.restype = ctypes.c_int64
    lib.msda_b200_launch_count.argtypes = [ctypes.c_int]
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
