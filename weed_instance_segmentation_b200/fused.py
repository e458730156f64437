"""Fused-prologue operator: softmax + sampling locations computed inside the MSDeformAttn kernels.

``ms_deform_attn_fused(value, value_spatial_shapes, level_start_index, sampling_offsets,
attention_logits, reference_points)`` replaces the block M2F:952-980 of the reference module
(``Mask2FormerPixelDecoderEncoderMultiscaleDeformableAttention.forward``):

    attention_weights  = softmax(attention_logits, -1)                        # M2F:955-960
    sampling_locations = reference_points[:, :, None, :, None, :]
                         + sampling_offsets / (W_l, H_l)                       # M2F:962-971
    output             = multi_scale_deformable_attention(value, shapes, sampling_locations,
                                                          attention_weights)   # M2F:980

in one kernel launch per direction (``msda_b200_forward_fused`` / ``msda_b200_backward_fused``), so
``sampling_locations`` (132 MB at BASELINE config 2) and ``attention_weights`` (33-66 MB) never go
through HBM, and the separate softmax / add / div kernels and their autograd nodes disappear.
Only the 2-coordinate reference-point form (M2F:962) is fused; reference points receive no gradient
(they are constants of the geometry, M2F:1095-1125).
"""
from __future__ import annotations

import torch

from . import _cabi
from . import functional as F

_DTYPE_CODE = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}


def _aux_dtype(value, offsets, logits):
    """dtype shared by offsets/logits inside the kernel: fp32 for fp32 values, else bf16 if both are bf16."""
    if value.dtype == torch.float32:
        return torch.float32
    if offsets.dtype == torch.bfloat16 and logits.dtype == torch.bfloat16:
        return torch.bfloat16
    return torch.float32


class MSDeformAttnFusedFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, value, shapes, level_start, offsets, logits, ref_points, query_order, want_attn):
        lib = _cabi.load()
        in_dtypes = (offsets.dtype, logits.dtype)
        aux = _aux_dtype(value, offsets, logits)
        value_c = value.contiguous()
        offsets_c = offsets.to(aux).contiguous()
        logits_c = logits.to(aux).contiguous()
        ref_c = ref_points.float().contiguous() if ref_points is not None else None  # None: computed in the kernels
        B, S, H, D = value_c.shape
        _, Q, _, L, P, _ = offsets_c.shape
        out = torch.empty((B, Q, H * D), dtype=value_c.dtype, device=value_c.device)
        attn = torch.empty((B, Q, H, L, P), dtype=torch.float32, device=value_c.device) if want_attn else None
        desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _DTYPE_CODE[value_c.dtype], _DTYPE_CODE[aux], shapes, level_start)
        with torch.cuda.device(value_c.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_forward_fused(desc, F._ptr(value_c), F._ptr(offsets_c), F._ptr(logits_c),
                                                    F._ptr(ref_c), F._ptr(out), F._ptr(attn), F._ptr(query_order), stream))
        ctx.save_for_backward(value_c, offsets_c, logits_c, ref_c, query_order)
        ctx.geom = (shapes, level_start, in_dtypes)
        del keep
        if want_attn:
            ctx.mark_non_differentiable(attn)
            return out, attn
        return out, None

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out, _grad_attn_unused):
        lib = _cabi.load()
        value, offsets, logits, ref, query_order = ctx.saved_tensors
        shapes, level_start, (off_dtype, logit_dtype) = ctx.geom
        B, S, H, D = value.shape
        _, Q, _, L, P, _ = offsets.shape
        flags = 0
        if F.deterministic():
            flags |= _cabi.FLAG_DETERMINISTIC
        else:
            if F._BF16_ATOMICS and value.dtype == torch.bfloat16:
                flags |= _cabi.FLAG_BF16_ATOMICS
            if F._BWD_V1:
                flags |= _cabi.FLAG_BWD_V1
        desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _DTYPE_CODE[value.dtype], _DTYPE_CODE[offsets.dtype],
                                     shapes, level_start, flags)
        grad_out = grad_out.to(value.dtype).contiguous()
        grad_value = torch.empty_like(value)
        grad_offsets = torch.empty_like(offsets)
        grad_logits = torch.empty_like(logits)
        ws_bytes = int(lib.msda_b200_backward_workspace_bytes(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=value.device) if ws_bytes else None
        with torch.cuda.device(value.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_backward_fused(desc, F._ptr(value), F._ptr(offsets), F._ptr(logits), F._ptr(ref),
                                                     F._ptr(grad_out), F._ptr(grad_value), F._ptr(grad_offsets),
                                                     F._ptr(grad_logits), F._ptr(ws), ws_bytes, F._ptr(query_order), stream))
        del keep
        if grad_offsets.dtype != off_dtype:
            grad_offsets = grad_offsets.to(off_dtype)
        if grad_logits.dtype != logit_dtype:
            grad_logits = grad_logits.to(logit_dtype)
        return grad_value, None, None, grad_offsets, grad_logits, None, None, None


def ms_deform_attn_fused(value, value_spatial_shapes, level_start_index, sampling_offsets, attention_logits,
                         reference_points, *, return_attention_weights: bool = False):
    """Fused softmax + sampling-location prologue + multi-scale deformable attention.

    Args:
        value: ``(B, S, H, D)`` float32 / bfloat16, CUDA.
        value_spatial_shapes: ``L`` pairs ``(H_l, W_l)``.
        level_start_index: ``(L,)`` or ``None`` (prefix sum of the shapes).
        sampling_offsets: ``(B, Q, H, L, P, 2)`` raw output of the ``sampling_offsets`` projection, in pixels.
        attention_logits: ``(B, Q, H, L*P)`` (or ``(B, Q, H, L, P)``) raw output of the ``attention_weights`` projection.
        reference_points: ``(B, Q, L, 2)`` normalised ``(x, y)`` (M2F:1095-1125), or ``None`` when ``Q == S`` (the pixel
            decoder's self-attention, query i = pixel i): the kernels then derive each query's reference point -- the
            centre of its own pixel, for every level -- from its index, exactly as ``get_reference_points`` does for
            un-padded inputs (``valid_ratios == 1``); no reference-point tensor is built or read.
    Returns:
        ``output (B, Q, H*D)`` and, if requested, ``attention_weights (B, Q, H, L, P)`` float32 (no gradient).
    """
    shapes = F._shapes_list(value_spatial_shapes)
    if not (value.is_cuda and sampling_offsets.is_cuda and attention_logits.is_cuda
            and (reference_points is None or reference_points.is_cuda)):
        raise RuntimeError("ms_deform_attn_fused: tensors must live on a CUDA device (this package has no CPU fallback)")
    if value.dim() != 4:
        raise ValueError(f"value must be (B, S, H, D), got {tuple(value.shape)}")
    if sampling_offsets.dim() != 6 or sampling_offsets.shape[-1] != 2:
        raise ValueError(f"sampling_offsets must be (B, Q, H, L, P, 2), got {tuple(sampling_offsets.shape)}")
    B, S, H, D = value.shape
    Bq, Q, Hq, L, P, _ = sampling_offsets.shape
    if (Bq, Hq) != (B, H) or len(shapes) != L:
        raise ValueError("sampling_offsets / spatial shapes do not match value")
    if attention_logits.numel() != B * Q * H * L * P or attention_logits.shape[:3] != (B, Q, H):
        raise ValueError(f"attention_logits must be {(B, Q, H, L * P)}, got {tuple(attention_logits.shape)}")
    if reference_points is None:
        if Q != S or Q != sum(h * w for h, w in shapes):
            raise ValueError("implicit reference points (reference_points=None) need Q == S == sum of the level sizes")
    else:
        if reference_points.shape[-1] != 2:
            raise ValueError(f"Last dim of reference_points must be 2 for the fused op, got {reference_points.shape[-1]}")
        if tuple(reference_points.shape) != (B, Q, L, 2):
            reference_points = reference_points.expand(B, Q, L, 2)
        if reference_points.requires_grad:
            raise ValueError("ms_deform_attn_fused does not differentiate with respect to reference_points")
    if sum(h * w for h, w in shapes) > S:
        raise ValueError(f"spatial shapes cover more rows than value has (S={S})")
    if value.dtype not in _DTYPE_CODE:
        raise TypeError(f"value dtype {value.dtype} unsupported (float32 or bfloat16)")
    level_start = F._level_start(shapes, level_start_index)
    order = None
    if F._USE_ORDER and Q == S and Q == sum(h * w for h, w in shapes) and level_start == F._level_start(shapes, None):
        order = F.query_order_2d(shapes, F._TILE, value.device)
    out, attn = MSDeformAttnFusedFunction.apply(value, shapes, level_start, sampling_offsets,
                                                attention_logits.reshape(B, Q, H, L * P), reference_points, order,
                                                return_attention_weights)
    return (out, attn) if return_attention_weights else out
