"""Projection with a fused bias-gradient reduction (SURVEY.md section 8(f) rank 2, encoder-layer epilogue).

``linear(x, weight, bias)`` is ``F.linear`` -- the GEMMs stay on cuBLAS tensor cores -- with one change in the
backward: ``grad_bias = grad_out.sum(rows)`` runs in ``msda_b200_column_sum`` (one streaming pass with 16-byte loads)
instead of torch's generic reduce kernel, which takes ~110 us per projection at BASELINE config 2 (six projections per
encoder layer). Under autocast the inputs are cast to the autocast dtype exactly as ``F.linear`` would.
"""
from __future__ import annotations

import os

import torch
import torch.nn.functional as F

from . import _cabi
from .functional import deterministic

_DTYPE_CODE = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}

# float32 projections on the bf16 tensor cores (csrc/gemm_f32.cu: cuBLASLt's CUBLAS_COMPUTE_32F_EMULATED_16BFX9, at least
# SGEMM's accuracy at ~2x its speed). MSDA_B200_F32_GEMM=native keeps torch's SGEMM.
_F32_EMULATED = os.environ.get("MSDA_B200_F32_GEMM", "emulated") != "native"
_f32_ws: dict = {}
_F32_WS_BYTES = 64 << 20


def f32_gemm_available() -> bool:
    """True when the CUDA toolkit's cuBLASLt (>= 12.9) could be opened and accepts the emulated float32 compute type."""
    return bool(_F32_EMULATED and torch.cuda.is_available() and _cabi.load().msda_b200_linear_f32_available())


def _use_f32_gemm(x, weight) -> bool:
    return (_F32_EMULATED and x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32
            and not torch.is_autocast_enabled("cuda") and x.numel() > 0 and not deterministic() and f32_gemm_available())


def _f32_workspace(device):
    ws = _f32_ws.get(device)
    if ws is None:
        ws = _f32_ws[device] = torch.empty(_F32_WS_BYTES, dtype=torch.uint8, device=device)
    return ws


def _f32_forward(x2, weight, bias, relu):
    lib = _cabi.load()
    y = torch.empty((x2.shape[0], weight.shape[0]), dtype=torch.float32, device=x2.device)
    ws = _f32_workspace(x2.device)
    with torch.cuda.device(x2.device):
        _cabi.check(lib.msda_b200_linear_f32_forward(x2.data_ptr(), weight.data_ptr(), bias.data_ptr() if bias is not None else None,
                                                     1 if relu else 0, y.data_ptr(), x2.shape[0], weight.shape[0], weight.shape[1],
                                                     ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream))
    return y


def _f32_backward(g2, x2, weight, need_x, need_w):
    lib = _cabi.load()
    ws = _f32_workspace(g2.device)
    M, N, K = g2.shape[0], weight.shape[0], weight.shape[1]
    gx = gw = None
    with torch.cuda.device(g2.device):
        stream = torch.cuda.current_stream().cuda_stream
        if need_x:
            gx = torch.empty((M, K), dtype=torch.float32, device=g2.device)
            _cabi.check(lib.msda_b200_linear_f32_grad_input(g2.data_ptr(), weight.data_ptr(), gx.data_ptr(), M, N, K,
                                                            ws.data_ptr(), ws.numel(), stream))
        if need_w:
            gw = torch.empty((N, K), dtype=torch.float32, device=g2.device)
            _cabi.check(lib.msda_b200_linear_f32_grad_weight(g2.data_ptr(), x2.data_ptr(), gw.data_ptr(), M, N, K,
                                                             ws.data_ptr(), ws.numel(), stream))
    return gx, gw


def column_sum(matrix: torch.Tensor) -> torch.Tensor:
    """``matrix.reshape(-1, C).sum(0)`` in float32 through the C ABI."""
    lib = _cabi.load()
    C = matrix.shape[-1]
    m = matrix.contiguous()
    out = torch.empty(C, dtype=torch.float32, device=m.device)
    with torch.cuda.device(m.device):
        _cabi.check(lib.msda_b200_column_sum(m.data_ptr() if m.numel() else None, _DTYPE_CODE[m.dtype], out.data_ptr(),
                                             m.numel() // C, C, torch.cuda.current_stream().cuda_stream))
    return out


def relu_backward_column_sum(grad_y: torch.Tensor, y: torch.Tensor):
    """``(threshold_backward(grad_y, y, 0), its sum over rows in float32)`` from one kernel: the FFN's ReLU backward and
    fc1's bias gradient. ``grad_y`` and ``y``: same shape / dtype (float32 or bfloat16), CUDA."""
    lib = _cabi.load()
    C = y.shape[-1]
    g, a = grad_y.contiguous(), y.contiguous()
    out = torch.empty_like(g)
    col = torch.empty(C, dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        _cabi.check(lib.msda_b200_relu_backward_column_sum(g.data_ptr() if g.numel() else None, a.data_ptr() if a.numel() else None,
                                                           _DTYPE_CODE[g.dtype], out.data_ptr() if out.numel() else None,
                                                           col.data_ptr(), g.numel() // C, C,
                                                           torch.cuda.current_stream().cuda_stream))
    return out, col


class LinearFunction(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, x, weight, bias):
        if torch.is_autocast_enabled("cuda"):
            dt = torch.get_autocast_dtype("cuda")
            xc, wc, bc = x.to(dt), weight.to(dt), bias.to(dt)
            with torch.autocast("cuda", enabled=False):
                y = F.linear(xc, wc, bc)
        else:
            xc, wc = x, weight
            ctx.f32 = _use_f32_gemm(x, weight) and bias.dtype == torch.float32
            if ctx.f32:
                xc, wc = x.contiguous(), weight.contiguous()
                y = _f32_forward(xc.reshape(-1, xc.shape[-1]), wc, bias.contiguous(), False).reshape(*xc.shape[:-1], wc.shape[0])
            else:
                y = F.linear(x, weight, bias)
        ctx.save_for_backward(xc, wc)
        ctx.in_dtypes = (x.dtype, weight.dtype, bias.dtype)
        return y

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, grad_y):
        xc, wc = ctx.saved_tensors
        xd, wd, bd = ctx.in_dtypes
        gy = grad_y.to(xc.dtype).contiguous()
        g2 = gy.reshape(-1, gy.shape[-1])
        need_x, need_w, need_b = ctx.needs_input_grad
        if getattr(ctx, "f32", False):
            grad_x, grad_w = _f32_backward(g2, xc.reshape(-1, xc.shape[-1]), wc, need_x, need_w)
            grad_x = grad_x.reshape(xc.shape) if need_x else None
        else:
            grad_x = (g2 @ wc).reshape(xc.shape).to(xd) if need_x else None
            grad_w = (g2.t() @ xc.reshape(-1, xc.shape[-1])).to(wd) if need_w else None
        grad_b = column_sum(g2).to(bd) if need_b else None
        return grad_x, grad_w, grad_b


class LinearReLUFunction(torch.autograd.Function):
    """``relu(F.linear(x, weight, bias))`` with bias + ReLU in the GEMM epilogue (cuBLASLt through
    ``torch._addmm_activation``; the GEMM stays a library call, M2F:1052-1053) and the bias gradient from the B200
    column-sum kernel."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, x, weight, bias):
        if torch.is_autocast_enabled("cuda"):
            dt = torch.get_autocast_dtype("cuda")
            xc, wc, bc = x.to(dt), weight.to(dt), bias.to(dt)
        else:
            xc, wc, bc = x, weight, bias
        ctx.f32 = (not torch.is_autocast_enabled("cuda")) and _use_f32_gemm(x, weight) and bias.dtype == torch.float32
        if ctx.f32:
            xc, wc = x.contiguous(), weight.contiguous()
            y = _f32_forward(xc.reshape(-1, xc.shape[-1]), wc, bias.contiguous(), True)
        else:
            with torch.autocast("cuda", enabled=False):
                y = torch._addmm_activation(bc, xc.reshape(-1, xc.shape[-1]), wc.t(), use_gelu=False)
        y = y.reshape(*xc.shape[:-1], wc.shape[0])
        ctx.save_for_backward(xc, wc, y)
        ctx.in_dtypes = (x.dtype, weight.dtype, bias.dtype)
        return y

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, grad_y):
        xc, wc, y = ctx.saved_tensors
        xd, wd, bd = ctx.in_dtypes
        # relu' and the bias gradient (the column sum of the masked gradient) from one pass over the matrix
        gy, col = relu_backward_column_sum(grad_y.to(y.dtype), y)
        g2 = gy.reshape(-1, gy.shape[-1])
        need_x, need_w, need_b = ctx.needs_input_grad
        if getattr(ctx, "f32", False):
            grad_x, grad_w = _f32_backward(g2, xc.reshape(-1, xc.shape[-1]), wc, need_x, need_w)
            grad_x = grad_x.reshape(xc.shape) if need_x else None
        else:
            grad_x = (g2 @ wc).reshape(xc.shape).to(xd) if need_x else None
            grad_w = (g2.t() @ xc.reshape(-1, xc.shape[-1])).to(wd) if need_w else None
        grad_b = col.to(bd) if need_b else None
        return grad_x, grad_w, grad_b


def _kernel_ok(x, weight, bias) -> bool:
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    C = weight.shape[0]
    return (x.is_cuda and bias is not None and dt in _DTYPE_CODE and C % (8 if dt == torch.bfloat16 else 4) == 0
            and C <= (2048 if dt == torch.bfloat16 else 1024))


def linear_relu(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``relu(F.linear(x, weight, bias))``, bias and ReLU in the GEMM epilogue (see :class:`LinearReLUFunction`)."""
    if not _kernel_ok(x, weight, bias):
        return F.relu(F.linear(x, weight, bias))
    return LinearReLUFunction.apply(x, weight, bias)


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``F.linear(x, weight, bias)`` whose backward reduces the bias gradient with the B200 kernel.

    Falls back to ``F.linear`` for shapes / dtypes the kernel does not cover (never for missing CUDA: there the
    call simply is ``F.linear``, which is what the reference does).
    """
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    C = weight.shape[0]
    ok = (x.is_cuda and bias is not None and dt in _DTYPE_CODE and C % (8 if dt == torch.bfloat16 else 4) == 0
          and C <= (2048 if dt == torch.bfloat16 else 1024))
    if not ok:
        return F.linear(x, weight, bias)
    return LinearFunction.apply(x, weight, bias)


class QueryValueCastFunction(torch.autograd.Function):
    """``(bfloat16(hidden + pos), bfloat16(hidden))`` in one pass (``msda_b200_query_value_cast_*``)."""

    @staticmethod
    def forward(ctx, hidden, pos):
        lib = _cabi.load()
        ctx.set_materialize_grads(False)
        h, p = hidden.contiguous(), pos.contiguous()
        q = torch.empty(h.shape, dtype=torch.bfloat16, device=h.device)
        v = torch.empty(h.shape, dtype=torch.bfloat16, device=h.device)
        with torch.cuda.device(h.device):
            _cabi.check(lib.msda_b200_query_value_cast_forward(h.data_ptr() if h.numel() else None,
                                                               p.data_ptr() if p.numel() else None,
                                                               q.data_ptr() if q.numel() else None,
                                                               v.data_ptr() if v.numel() else None, h.numel(),
                                                               torch.cuda.current_stream().cuda_stream))
        ctx.shape, ctx.device = h.shape, h.device
        return q, v

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_q, grad_v):
        lib = _cabi.load()
        need_h, need_p = ctx.needs_input_grad
        if not (need_h or need_p):
            return None, None
        gq = grad_q.to(torch.bfloat16).contiguous() if grad_q is not None else None
        gv = grad_v.to(torch.bfloat16).contiguous() if grad_v is not None else None
        gh = torch.empty(ctx.shape, dtype=torch.float32, device=ctx.device)
        gp = torch.empty(ctx.shape, dtype=torch.float32, device=ctx.device) if need_p else None
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
        with torch.cuda.device(ctx.device):
            _cabi.check(lib.msda_b200_query_value_cast_backward(ptr(gq), ptr(gv), ptr(gh), ptr(gp), gh.numel(),
                                                                torch.cuda.current_stream().cuda_stream))
        return (gh if need_h else None), gp


def query_value_cast(hidden: torch.Tensor, pos: torch.Tensor):
    """The attention module's two bfloat16 operands from the float32 hidden state and position embedding
    (M2F:936-937, 947): ``(bfloat16(hidden + pos), bfloat16(hidden))``, one kernel per direction instead of an fp32 add and
    two casts (forward) / two casts and an add (backward). Same values as the stock sequence."""
    if not (hidden.is_cuda and pos.is_cuda):
        raise RuntimeError("query_value_cast: tensors must live on a CUDA device (this package has no CPU fallback)")
    if hidden.dtype != torch.float32 or pos.dtype != torch.float32:
        raise TypeError("query_value_cast: float32 inputs only")
    if hidden.shape != pos.shape:
        raise ValueError(f"query_value_cast: hidden {tuple(hidden.shape)} and pos {tuple(pos.shape)} differ")
    if hidden.numel() % 8:
        raise ValueError("query_value_cast: the element count must be a multiple of 8")
    return QueryValueCastFunction.apply(hidden, pos)
