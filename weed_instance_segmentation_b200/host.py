"""The operator for callers whose tensors live in HOST memory (``msda_b200_host_pipeline_*`` in the C ABI).

``HostPipeline`` takes CPU tensors in the operator's layouts (M2F:798-837 arguments plus ``grad_output``), streams
them through the device image by image -- H2D copy, forward (+ backward) kernels and D2H copy overlap on three
streams -- and writes the results into caller-provided CPU tensors. Pinned (page-locked) tensors are needed for
the copies to overlap; pageable ones work but serialise. There is no CPU compute path: the arithmetic is the same
CUDA kernels ``ms_deform_attn`` launches.
"""
from __future__ import annotations

import ctypes
from typing import Sequence

import torch

from . import _cabi, functional

_DTYPE_CODE = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}


class HostPipeline:
    """Forward (+ backward) of MSDeformAttn over host buffers for a fixed problem geometry.

    ``batch`` images per step, ``num_queries`` queries per image (``None``: one query per pixel),
    ``chunk_images`` images per staging chunk, ``slots`` staging slots (device memory: ``slots`` chunks).
    ``deterministic``: run the backward with ``FLAG_DETERMINISTIC`` (bit-identical gradients for identical inputs,
    whatever the chunking); ``None`` follows ``torch.use_deterministic_algorithms`` at construction.
    """

    def __init__(self, batch: int, spatial_shapes: Sequence[tuple[int, int]], num_heads: int, head_dim: int,
                 num_points: int, value_dtype: torch.dtype = torch.bfloat16, attn_dtype: torch.dtype | None = None,
                 num_queries: int | None = None, backward: bool = True, chunk_images: int = 1, slots: int = 3,
                 device: torch.device | int | None = None, deterministic: bool | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("HostPipeline needs a CUDA device (this package has no CPU fallback)")
        self._handle = None
        self._lib = _cabi.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.shapes = [(int(h), int(w)) for h, w in spatial_shapes]
        self.B, self.H, self.D, self.P, self.L = int(batch), int(num_heads), int(head_dim), int(num_points), len(self.shapes)
        self.S = sum(h * w for h, w in self.shapes)
        self.Q = self.S if num_queries is None else int(num_queries)
        self.value_dtype = value_dtype
        self.attn_dtype = value_dtype if attn_dtype is None else attn_dtype
        if self.value_dtype not in _DTYPE_CODE or self.attn_dtype not in _DTYPE_CODE:
            raise TypeError("HostPipeline: float32 or bfloat16 tensors only")
        self.backward = bool(backward)
        self.deterministic = functional.deterministic() if deterministic is None else bool(deterministic)
        flags = 0
        if self.deterministic:
            flags |= _cabi.FLAG_DETERMINISTIC
        else:
            if functional._BF16_ATOMICS and value_dtype == torch.bfloat16:
                flags |= _cabi.FLAG_BF16_ATOMICS
            if functional._BWD_V1:
                flags |= _cabi.FLAG_BWD_V1
        lsi = functional._level_start(self.shapes, None)
        desc, self._keep = _cabi.make_desc(self.B, self.S, self.Q, self.H, self.D, self.L, self.P,
                                           _DTYPE_CODE[self.value_dtype], _DTYPE_CODE[self.attn_dtype], self.shapes, lsi,
                                           flags)
        # the 2-D query order is a scheduling hint for one-query-per-pixel problems (functional.query_order_2d)
        self._order = (functional.query_order_2d(self.shapes, functional._TILE, self.device)
                       if functional._USE_ORDER and self.Q == self.S else None)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.msda_b200_host_pipeline_create(
                ctypes.byref(desc), int(chunk_images), int(slots), int(self.backward),
                self._order.data_ptr() if self._order is not None else None, ctypes.byref(handle)))
        self._handle = handle
        LP2 = (self.H, self.L, self.P)
        self._in_spec = {
            "value": ((self.B, self.S, self.H, self.D), self.value_dtype),
            "sampling_locations": ((self.B, self.Q, *LP2, 2), torch.float32),
            "attention_weights": ((self.B, self.Q, *LP2), self.attn_dtype),
            "grad_output": ((self.B, self.Q, self.H * self.D), self.value_dtype),
        }
        self._out_spec = {
            "output": self._in_spec["grad_output"],
            "grad_value": self._in_spec["value"],
            "grad_sampling_locations": self._in_spec["sampling_locations"],
            "grad_attention_weights": self._in_spec["attention_weights"],
        }

    # ------------------------------------------------------------------ buffers
    def empty_outputs(self, pin: bool = True) -> dict[str, torch.Tensor]:
        """Host tensors of the right shapes / dtypes for ``step``'s results."""
        names = list(self._out_spec) if self.backward else ["output"]
        return {n: torch.empty(self._out_spec[n][0], dtype=self._out_spec[n][1], pin_memory=pin) for n in names}

    def _check(self, name, t, spec):
        shape, dtype = spec
        if not isinstance(t, torch.Tensor) or t.is_cuda:
            raise RuntimeError(f"HostPipeline: {name} must be a CPU tensor (device tensors go through ms_deform_attn)")
        if t.dtype != dtype:
            raise TypeError(f"HostPipeline: {name} has dtype {t.dtype}, expected {dtype}")
        if t.numel() != _numel(shape) or (t.dim() == len(shape) and tuple(t.shape) != tuple(shape)):
            raise ValueError(f"HostPipeline: {name} has shape {tuple(t.shape)}, expected {tuple(shape)}")
        if not t.is_contiguous():
            raise ValueError(f"HostPipeline: {name} must be contiguous")
        return t.data_ptr()

    # ------------------------------------------------------------------ the call
    def step(self, value, sampling_locations, attention_weights, grad_output=None, *, output, grad_value=None,
             grad_sampling_locations=None, grad_attention_weights=None, stream: torch.cuda.Stream | None = None) -> None:
        """Enqueue one batch; returns without waiting. Results are valid after ``join()`` + a synchronise of the
        stream (or after ``synchronize()``); keep every tensor alive and untouched until then."""
        if self._handle is None:
            raise RuntimeError("HostPipeline: closed")
        ins = {"value": value, "sampling_locations": sampling_locations, "attention_weights": attention_weights}
        outs = {"output": output}
        if self.backward:
            ins["grad_output"] = grad_output
            outs.update(grad_value=grad_value, grad_sampling_locations=grad_sampling_locations,
                        grad_attention_weights=grad_attention_weights)
        ptr = {n: self._check(n, t, self._in_spec[n]) for n, t in ins.items()}
        ptr.update({n: self._check(n, t, self._out_spec[n]) for n, t in outs.items()})
        with torch.cuda.device(self.device):
            st = (stream or torch.cuda.current_stream()).cuda_stream
            _cabi.check(self._lib.msda_b200_host_pipeline_step(
                self._handle, ptr["value"], ptr["sampling_locations"], ptr["attention_weights"], ptr.get("grad_output"),
                ptr["output"], ptr.get("grad_value"), ptr.get("grad_sampling_locations"),
                ptr.get("grad_attention_weights"), st))

    def join(self, stream: torch.cuda.Stream | None = None) -> None:
        """Make ``stream`` (default: the current one) wait for everything enqueued so far."""
        with torch.cuda.device(self.device):
            st = (stream or torch.cuda.current_stream()).cuda_stream
            _cabi.check(self._lib.msda_b200_host_pipeline_join(self._handle, st))

    def synchronize(self) -> None:
        _cabi.check(self._lib.msda_b200_host_pipeline_sync(self._handle))

    @property
    def h2d_bytes_per_step(self) -> int:
        names = list(self._in_spec) if self.backward else list(self._in_spec)[:3]
        return sum(_numel(self._in_spec[n][0]) * _itemsize(self._in_spec[n][1]) for n in names)

    @property
    def d2h_bytes_per_step(self) -> int:
        names = list(self._out_spec) if self.backward else ["output"]
        return sum(_numel(self._out_spec[n][0]) * _itemsize(self._out_spec[n][1]) for n in names)

    def close(self) -> None:
        if self._handle is not None:
            self._lib.msda_b200_host_pipeline_destroy(self._handle)
            self._handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _numel(shape) -> int:
    n = 1
    for v in shape:
        n *= int(v)
    return n


def _itemsize(dtype) -> int:
    return 2 if dtype == torch.bfloat16 else 4
