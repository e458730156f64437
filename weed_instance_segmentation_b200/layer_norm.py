"""Fused residual-add + LayerNorm for the pixel-decoder encoder layer (SURVEY.md section 8(f) rank 2).

``add_layer_norm(x, residual, weight, bias, eps)`` computes ``F.layer_norm(residual + x, (C,), weight, bias, eps)``
-- the two lines M2F:1049-1050 (and M2F:1058-1059) -- in one kernel per direction
(``csrc/layer_epilogue.cu``). The output is float32, which is what ``F.layer_norm`` returns under autocast; ``x`` is
typically the bfloat16 output of a projection and ``residual`` the float32 hidden state.
"""
from __future__ import annotations

import torch

from . import _cabi
from ._cabi import DTYPE_CODE, ptr


class AddLayerNormFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, residual, weight, bias, eps, also_lowp=False, clamp=None):
        lib = _cabi.load()
        ctx.set_materialize_grads(False)
        C = x.shape[-1]
        xc, rc = x.contiguous(), residual.contiguous()
        w, b = weight.float().contiguous(), bias.float().contiguous()
        rows = xc.numel() // C
        y = torch.empty(xc.shape, dtype=torch.float32, device=xc.device)
        mean = torch.empty(rows, dtype=torch.float32, device=xc.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=xc.device)
        y_lowp = torch.empty(xc.shape, dtype=torch.bfloat16, device=xc.device) if also_lowp else None
        with torch.cuda.device(xc.device):
            stream = torch.cuda.current_stream().cuda_stream
            if clamp is None:
                _cabi.check(lib.msda_b200_add_layernorm_forward(ptr(xc), DTYPE_CODE[xc.dtype], ptr(rc),
                                                                DTYPE_CODE[rc.dtype], ptr(w), ptr(b), float(eps), ptr(y),
                                                                ptr(y_lowp), ptr(mean), ptr(rstd), rows, C, stream))
            else:
                _cabi.check(lib.msda_b200_add_layernorm_clamp_forward(ptr(xc), DTYPE_CODE[xc.dtype], ptr(rc),
                                                                      DTYPE_CODE[rc.dtype], ptr(w), ptr(b), float(eps),
                                                                      float(clamp), ptr(y), ptr(y_lowp), ptr(mean),
                                                                      ptr(rstd), rows, C, stream))
        ctx.clamp = clamp
        ctx.save_for_backward(xc, rc, w, mean, rstd, *((b,) if clamp is not None else ()))
        ctx.param_dtypes = (weight.dtype, bias.dtype)
        return (y, y_lowp) if also_lowp else y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y, grad_y_lowp=None):
        lib = _cabi.load()
        x, r, w, mean, rstd = ctx.saved_tensors[:5]
        C = x.shape[-1]
        rows = x.numel() // C
        if grad_y is None:  # only the bfloat16 copy was used downstream
            grad_y, grad_y_lowp = grad_y_lowp.float(), None
        gy = grad_y.float().contiguous()
        gyl = grad_y_lowp.to(torch.bfloat16).contiguous() if grad_y_lowp is not None else None
        ds = torch.empty(x.shape, dtype=torch.float32, device=x.device)
        need_lowp = x.dtype == torch.bfloat16 or r.dtype == torch.bfloat16
        ds_lowp = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if need_lowp else None
        gw = torch.empty(C, dtype=torch.float32, device=x.device)
        gb = torch.empty(C, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            if ctx.clamp is None:
                _cabi.check(lib.msda_b200_add_layernorm_backward(ptr(gy), ptr(gyl), ptr(x), DTYPE_CODE[x.dtype], ptr(r),
                                                                 DTYPE_CODE[r.dtype], ptr(w), ptr(mean), ptr(rstd),
                                                                 ptr(ds), ptr(ds_lowp), ptr(gw), ptr(gb), rows, C, stream))
            else:
                _cabi.check(lib.msda_b200_add_layernorm_clamp_backward(
                    ptr(gy), ptr(gyl), ptr(x), DTYPE_CODE[x.dtype], ptr(r), DTYPE_CODE[r.dtype], ptr(w),
                    ptr(ctx.saved_tensors[5]), float(ctx.clamp), ptr(mean), ptr(rstd), ptr(ds), ptr(ds_lowp), ptr(gw),
                    ptr(gb), rows, C, stream))
        gx = ds_lowp if x.dtype == torch.bfloat16 else ds
        gr = ds_lowp if r.dtype == torch.bfloat16 else ds
        wd, bd = ctx.param_dtypes
        return gx, gr, gw.to(wd), gb.to(bd), None, None, None


def add_layer_norm(x: torch.Tensor, residual: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor,
                   eps: float = 1e-5, also_lowp: bool = False, clamp: float | None = None):
    """``F.layer_norm(residual + x, (C,), weight, bias, eps)`` in one kernel; float32 output.

    ``also_lowp``: additionally return the same values rounded to bfloat16 (``(y, y_bf16)``): the operand of the
    projection that follows under autocast, written by the same kernel instead of a separate cast; the gradient that
    returns through it is added inside the backward kernel.

    ``clamp``: fold ``torch.clamp(y, -clamp, clamp)`` (the encoder layer's closing clamp, M2F:1062-1065) into the same
    kernels, forward and backward, with torch.clamp's semantics (NaN stays NaN; no gradient where y is out of range).

    ``x`` and ``residual``: same shape ``(..., C)``, float32 or bfloat16, CUDA; ``C`` a multiple of 128, at most 512.
    """
    if not (x.is_cuda and residual.is_cuda):
        raise RuntimeError("add_layer_norm: tensors must live on a CUDA device (this package has no CPU fallback)")
    if x.shape != residual.shape:
        raise ValueError(f"add_layer_norm: x {tuple(x.shape)} and residual {tuple(residual.shape)} differ")
    if x.dtype not in DTYPE_CODE or residual.dtype not in DTYPE_CODE:
        raise TypeError("add_layer_norm: float32 or bfloat16 inputs only")
    C = x.shape[-1]
    if weight.numel() != C or bias.numel() != C:
        raise ValueError("add_layer_norm: weight / bias must have C elements")
    if clamp is not None and not clamp > 0:
        raise ValueError("add_layer_norm: clamp must be positive")
    return AddLayerNormFunction.apply(x, residual, weight, bias, eps, also_lowp, clamp)
