"""Host side of the MSDeformAttn operator: the reference's call signature over the C ABI.

``ms_deform_attn(value, value_spatial_shapes, level_start_index, sampling_locations,
attention_weights)`` keeps the five-tensor operator signature of the original Deformable-DETR
CUDA op (``MSDeformAttnFunction.apply``; the argument order HF preserves at
``transformers/models/deformable_detr/modeling_deformable_detr.py:171-181``), and
``multi_scale_deformable_attention(value, value_spatial_shapes, sampling_locations,
attention_weights)`` is the four-argument form Mask2Former calls
(``transformers/models/mask2former/modeling_mask2former.py:798-837`` defined, ``:980`` called).

PyTorch is plumbing here (device memory, streams, autograd bookkeeping); all arithmetic runs in
``libmsda_b200.so`` (``csrc/msda_b200.cu``). There is no CPU path and no PyTorch fallback:
non-CUDA tensors raise.

Error behaviour mirrors the reference module (M2F:942-945, :978): shape mismatches raise
``ValueError``; failures inside the library raise ``MSDAError`` (never swallowed).
"""
from __future__ import annotations

import os
import weakref
from typing import Sequence

import torch

from . import _cabi
from ._cabi import MSDAError  # noqa: F401  (re-export)

_DTYPE_CODE = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}

# Scheduling knobs (results never depend on them).
def _parse_tile(text):
    parts = [int(v) for v in text.lower().split("x")]
    return (parts[0], parts[0]) if len(parts) == 1 else (parts[0], parts[1])


# 2-D query tile (rows x cols) of the query order. The pixel-sorted backward (csrc/msda_bwd_sorted.cuh) owns 128
# queries per block; an 8 x 16 patch keeps their samples inside a small pixel window, which is what lets it merge
# contributions before reducing. The forward does not care (measured: LSU-bound either way, profiles/r01_notes.md).
_TILE = _parse_tile(os.environ.get("MSDA_B200_TILE", "8x16"))
_USE_ORDER = os.environ.get("MSDA_B200_QUERY_ORDER", "1") != "0"
_BF16_ATOMICS = os.environ.get("MSDA_B200_BF16_ATOMICS", "0") == "1"
_BWD_V1 = os.environ.get("MSDA_B200_BWD_V1", "0") == "1"
_BWD_V2 = os.environ.get("MSDA_B200_BWD_V2", "0") == "1"  # CUDA-core pixel-sorted backward instead of the tensor-core one
# Forward: never multiply a zero-weight corner (exact zeros padding even when `value` holds NaN / Inf in pixels no
# sample reads; 25-30 % slower, see include/msda_b200.h MSDA_B200_FLAG_STRICT_PADDING).
_STRICT_PADDING = os.environ.get("MSDA_B200_STRICT_PADDING", "0") == "1"

_order_cache: dict = {}
_lsi_checked: dict = {}


def _shapes_list(value_spatial_shapes) -> list[tuple[int, int]]:
    """``spatial_shapes_list`` (M2F:1312) as host ints. A CUDA tensor costs one sync; pass a list."""
    if isinstance(value_spatial_shapes, torch.Tensor):
        value_spatial_shapes = value_spatial_shapes.tolist()
    return [(int(h), int(w)) for h, w in value_spatial_shapes]


def _level_start(shapes: Sequence[tuple[int, int]], level_start_index) -> list[int]:
    """Host copy of ``level_start_index`` (M2F:1321).

    HF threads a CUDA tensor through every layer but the reference op never reads it. Reading it back costs a device
    sync, so the host copy is remembered per tensor object (the same tensor reaches all six layers of a forward).
    """
    derived, acc = [], 0
    for h, w in shapes:
        derived.append(acc)
        acc += h * w
    if level_start_index is None:
        return derived
    if isinstance(level_start_index, torch.Tensor):
        if level_start_index.is_cuda:
            # keyed on the tensor OBJECT and its version counter (not on data_ptr: the caching allocator hands the same
            # address to later tensors with other contents); HF builds a fresh tensor per forward, so in practice this
            # costs one small D2H read per forward of the model, not per layer
            key = (tuple(shapes), id(level_start_index), level_start_index._version)
            hit = _lsi_checked.get(key)
            if hit is not None and hit[0]() is level_start_index:
                return hit[1]
            given = [int(v) for v in level_start_index.tolist()]
            if len(_lsi_checked) > 64:
                _lsi_checked.clear()
            _lsi_checked[key] = (weakref.ref(level_start_index), given)
            return given
        return [int(v) for v in level_start_index.tolist()]
    return [int(v) for v in level_start_index]


def query_order_2d(shapes: Sequence[tuple[int, int]], tile: int, device) -> torch.Tensor:
    """Permutation of 0..S-1 that walks every level in ``tile`` = (rows, cols) blocks (row-major inside).

    Used when ``Q == S`` (pixel-decoder self-attention: query i sits on pixel i, M2F:1117-1123):
    a thread block then owns a compact 2-D patch of queries whose samples overlap, which is what
    keeps the bilinear footprint in L1. Scheduling only; results do not depend on it.
    """
    th, tw = (tile, tile) if isinstance(tile, int) else tile
    key = (tuple(shapes), th, tw, str(device))
    hit = _order_cache.get(key)
    if hit is not None:
        return hit
    parts, start = [], 0
    for h, w in shapes:
        y = torch.arange(h).view(h, 1).expand(h, w)
        x = torch.arange(w).view(1, w).expand(h, w)
        tiles_x = (w + tw - 1) // tw
        rank = ((y // th) * tiles_x + (x // tw)) * (th * tw) + (y % th) * tw + (x % tw)
        parts.append(start + torch.argsort(rank.reshape(-1), stable=True))
        start += h * w
    order = torch.cat(parts).to(torch.int32).to(device)
    _order_cache[key] = order
    return order


def _check_inputs(value, shapes, loc, attn):
    if not (value.is_cuda and loc.is_cuda and attn.is_cuda):
        raise RuntimeError("ms_deform_attn: tensors must live on a CUDA device (this package has no CPU fallback)")
    if value.dim() != 4:
        raise ValueError(f"value must be (B, S, H, D), got {tuple(value.shape)}")
    if loc.dim() != 6 or loc.shape[-1] != 2:
        raise ValueError(f"sampling_locations must be (B, Q, H, L, P, 2), got {tuple(loc.shape)}")
    B, S, H, D = value.shape
    Bq, Q, Hq, L, P, _ = loc.shape
    if Bq != B or Hq != H:
        raise ValueError(f"sampling_locations {tuple(loc.shape)} does not match value {tuple(value.shape)}")
    if tuple(attn.shape) != (B, Q, H, L, P):
        raise ValueError(f"attention_weights must be {(B, Q, H, L, P)}, got {tuple(attn.shape)}")
    if len(shapes) != L:
        raise ValueError(f"{len(shapes)} spatial shapes for {L} levels")
    total = sum(h * w for h, w in shapes)
    if total > S:
        # M2F:942-945 ("Make sure to align the spatial shapes with the sequence length ...")
        raise ValueError(f"spatial shapes cover {total} rows but value has S={S}")
    if value.dtype not in _DTYPE_CODE:
        raise TypeError(f"value dtype {value.dtype} unsupported (float32 or bfloat16)")
    return B, S, Q, H, D, L, P


def _prepare(value, loc, attn):
    """Contiguity and dtype contract: loc fp32; attn fp32 for fp32 values, fp32 or bf16 for bf16 values."""
    value = value.contiguous()
    loc = loc.contiguous() if loc.dtype == torch.float32 else loc.float().contiguous()
    if value.dtype == torch.float32 and attn.dtype != torch.float32:
        attn = attn.float()
    elif attn.dtype not in _DTYPE_CODE:
        attn = attn.to(value.dtype)
    return value, loc, attn.contiguous()


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


class MSDeformAttnFunction(torch.autograd.Function):
    """Forward / backward through ``msda_b200_forward`` / ``msda_b200_backward``."""

    @staticmethod
    def forward(ctx, value, shapes, level_start, loc, attn, query_order, flags):
        lib = _cabi.load()
        in_dtypes = (loc.dtype, attn.dtype)
        value_c, loc_c, attn_c = _prepare(value, loc, attn)
        B, S, H, D = value_c.shape
        _, Q, _, L, P, _ = loc_c.shape
        out = torch.empty((B, Q, H * D), dtype=value_c.dtype, device=value_c.device)
        desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _DTYPE_CODE[value_c.dtype], _DTYPE_CODE[attn_c.dtype],
                                     shapes, level_start, flags)
        with torch.cuda.device(value_c.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_forward(desc, _ptr(value_c), _ptr(loc_c), _ptr(attn_c), _ptr(out),
                                              _ptr(query_order), stream))
        ctx.save_for_backward(value_c, loc_c, attn_c, query_order)
        ctx.geom = (shapes, level_start, flags, in_dtypes)
        del keep
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _cabi.load()
        value, loc, attn, query_order = ctx.saved_tensors
        shapes, level_start, flags, (loc_dtype, attn_dtype) = ctx.geom
        B, S, H, D = value.shape
        _, Q, _, L, P, _ = loc.shape
        grad_out = grad_out.to(value.dtype).contiguous()
        if _BF16_ATOMICS and value.dtype == torch.bfloat16:
            flags |= _cabi.FLAG_BF16_ATOMICS
        if _BWD_V1:
            flags |= _cabi.FLAG_BWD_V1
        if _BWD_V2:
            flags |= _cabi.FLAG_BWD_V2
        desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _DTYPE_CODE[value.dtype], _DTYPE_CODE[attn.dtype],
                                     shapes, level_start, flags)
        grad_value = torch.empty_like(value)
        grad_loc = torch.empty_like(loc)
        grad_attn = torch.empty_like(attn)
        ws_bytes = int(lib.msda_b200_backward_workspace_bytes(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=value.device) if ws_bytes else None
        with torch.cuda.device(value.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_backward(desc, _ptr(value), _ptr(loc), _ptr(attn), _ptr(grad_out),
                                               _ptr(grad_value), _ptr(grad_loc), _ptr(grad_attn),
                                               _ptr(ws), ws_bytes, _ptr(query_order), stream))
        del keep
        if grad_loc.dtype != loc_dtype:
            grad_loc = grad_loc.to(loc_dtype)
        if grad_attn.dtype != attn_dtype:
            grad_attn = grad_attn.to(attn_dtype)
        return grad_value, None, None, grad_loc, grad_attn, None, None


def ms_deform_attn(
    value: torch.Tensor,
    value_spatial_shapes,
    level_start_index,
    sampling_locations: torch.Tensor,
    attention_weights: torch.Tensor,
    *,
    profile: bool = False,
) -> torch.Tensor:
    """Multi-scale deformable attention, five-tensor operator signature.

    Args:
        value: ``(B, S, H, D)`` float32 or bfloat16 on a CUDA device.
        value_spatial_shapes: ``L`` pairs ``(H_l, W_l)`` (list of tuples as HF passes, or a tensor).
        level_start_index: ``(L,)`` first row of each level in ``S``; ``None`` = prefix sum of shapes.
        sampling_locations: ``(B, Q, H, L, P, 2)``, last dim ``(x, y)`` normalised to ``[0, 1]``.
        attention_weights: ``(B, Q, H, L, P)`` post-softmax.
    Returns:
        ``(B, Q, H*D)`` in ``value.dtype`` -- the same tensor M2F:798-837 returns.
    """
    shapes = _shapes_list(value_spatial_shapes)
    B, S, Q, H, D, L, P = _check_inputs(value, shapes, sampling_locations, attention_weights)
    level_start = _level_start(shapes, level_start_index)
    order = None
    if _USE_ORDER and Q == S and Q == sum(h * w for h, w in shapes) and level_start == _level_start(shapes, None):
        order = query_order_2d(shapes, _TILE, value.device)
    flags = _cabi.FLAG_PROFILE if profile else 0
    if _STRICT_PADDING:
        flags |= _cabi.FLAG_STRICT_PADDING
    return MSDeformAttnFunction.apply(value, shapes, level_start, sampling_locations, attention_weights, order, flags)


def multi_scale_deformable_attention(value, value_spatial_shapes, sampling_locations, attention_weights):
    """Drop-in for ``transformers...modeling_mask2former.multi_scale_deformable_attention`` (M2F:798)."""
    return ms_deform_attn(value, value_spatial_shapes, None, sampling_locations, attention_weights)
