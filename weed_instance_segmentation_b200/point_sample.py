"""Batched bilinear point sampling over planes that stay where they are (SURVEY.md section 8(f) rank 4).

The reference's ``sample_point`` (M2F:245-274) is ``grid_sample`` on a ``(R, 1, h, w)`` tensor, which forces the
callers to gather / pad / upcast the masks into such a tensor first (M2F:455-474, :689-705). ``point_sample`` takes
the original tensors and a per-row address instead::

    out[r, k] = bilinear(sources[src_id[r]][plane_id[r]], coords[coord_row[r], k])        # (R, K) float32

with ``grid_sample``'s conventions (bilinear, zeros padding, ``align_corners=False``, coordinates in [0, 1] as (x, y)).
Gradients flow to the sources that require them (scatter with fp32 atomics; under
``torch.use_deterministic_algorithms(True)`` a sort by destination pixel and ordered fp32 sums instead, so they are
bit-identical run to run); coordinates carry none.
CUDA only: ``csrc/point_sample.cu`` through the C ABI, no CPU path.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from . import _cabi
from .functional import deterministic

_DTYPE_CODE = {**_cabi.DTYPE_CODE, torch.uint8: _cabi.U8, torch.bool: _cabi.U8}


class _Rows:
    """Host-built address tables of one call (kept for the backward)."""

    def __init__(self, sources: Sequence[torch.Tensor], src_id, plane_id, coord_row, device):
        src_id = np.asarray(src_id, dtype=np.int64).reshape(-1)
        plane_id = np.asarray(plane_id, dtype=np.int64).reshape(-1)
        coord_row = np.asarray(coord_row, dtype=np.int64).reshape(-1)
        if not (src_id.shape == plane_id.shape == coord_row.shape):
            raise ValueError("point_sample: src_id, plane_id and coord_row must have one entry per row")
        self.R = int(src_id.shape[0])
        self.src_id, self.plane_id = src_id, plane_id
        n = np.array([s.shape[0] for s in sources], dtype=np.int64)
        self.h = np.array([s.shape[1] for s in sources], dtype=np.int64)
        self.w = np.array([s.shape[2] for s in sources], dtype=np.int64)
        if self.R:
            if src_id.min() < 0 or src_id.max() >= len(sources):
                raise ValueError("point_sample: src_id out of range")
            if plane_id.min() < 0 or (plane_id >= n[src_id]).any():
                raise ValueError("point_sample: plane_id out of range for its source")
        base = np.array([s.data_ptr() for s in sources], dtype=np.int64)
        item = np.array([s.element_size() for s in sources], dtype=np.int64)
        code = np.array([_DTYPE_CODE[s.dtype] for s in sources], dtype=np.int64)
        ptr = base[src_id] + plane_id * (self.h * self.w * item)[src_id]
        rows = np.stack([self.h[src_id], self.w[src_id], coord_row, code[src_id]], axis=1).astype(np.int32)
        self.device = device
        self.ptr = torch.from_numpy(ptr).to(device, non_blocking=True)
        self.rows_host = np.ascontiguousarray(rows)
        self.rows = torch.from_numpy(self.rows_host).to(device, non_blocking=True)
        self.max_coord_row = int(coord_row.max()) if self.R else -1

    def grad_pointers(self, grads: Sequence[torch.Tensor | None]) -> torch.Tensor:
        base = np.array([g.data_ptr() if g is not None else 0 for g in grads], dtype=np.int64)
        live = base[self.src_id] != 0
        ptr = np.where(live, base[self.src_id] + self.plane_id * (self.h * self.w * 4)[self.src_id], 0)
        return torch.from_numpy(ptr).to(self.device, non_blocking=True)

    def det_tables(self, grads: Sequence[torch.Tensor | None]):
        """Tables of the deterministic backward: the rows whose source has a gradient (``live``, host indices), their
        gradient-plane pointers, rows and destination keys (``key_base`` per row and the key count, see
        ``msda_b200_point_sample_backward_det``). Every distinct (source, plane) gets its own key range."""
        has = np.array([g is not None for g in grads])
        live = np.nonzero(has[self.src_id])[0]
        src, plane = self.src_id[live], self.plane_id[live]
        pairs, inverse = np.unique(np.stack([src, plane], axis=1), axis=0, return_inverse=True)
        size = (self.h * self.w)[pairs[:, 0]]
        start = np.concatenate([[0], np.cumsum(size)[:-1]]).astype(np.int64)
        key_base = start[inverse.reshape(-1)]
        base = np.array([g.data_ptr() if g is not None else 0 for g in grads], dtype=np.int64)
        ptr = base[src] + plane * (self.h * self.w * 4)[src]
        to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.device, non_blocking=True)
        return live, to_dev(ptr), to_dev(self.rows_host[live]), to_dev(key_base), int(size.sum())


class PointSampleFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, coords, table, *sources):
        lib = _cabi.load()
        K = coords.shape[1]
        out = torch.empty((table.R, K), dtype=torch.float32, device=coords.device)
        with torch.cuda.device(coords.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_point_sample_forward(_cabi.ptr(table.ptr), _cabi.ptr(table.rows),
                                                           _cabi.ptr(coords), _cabi.ptr(out), table.R, K, stream))
        ctx.table = table
        ctx.save_for_backward(coords)
        ctx.src_meta = [(s.shape, s.dtype) for s in sources]
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _cabi.load()
        (coords,) = ctx.saved_tensors
        table = ctx.table
        K = coords.shape[1]
        needs = ctx.needs_input_grad[2:]
        # Peak memory: one fp32 gradient per differentiable source is alive at once (the node returns them together) --
        # for the batched criterion that is all L decoder layers' (B*Q, h, w) logits, 0.2 GB per layer at batch 8 x 100
        # queries x 256^2 (2.1 GB for 10 layers), plus a transient low-precision copy per bf16 source. The reference's
        # per-layer index backward holds one layer at a time; on a 180 GB B200 the single launch is the better trade.
        grads = [torch.zeros(shape, dtype=torch.float32, device=coords.device) if need else None
                 for (shape, _), need in zip(ctx.src_meta, needs)]
        if table.R and K and any(needs):
            go = grad_out.float().contiguous()
            with torch.cuda.device(coords.device):
                stream = torch.cuda.current_stream().cuda_stream
                if deterministic():
                    _backward_det(lib, table, grads, coords, go, K, stream)
                else:
                    gptr = table.grad_pointers(grads)
                    _cabi.check(lib.msda_b200_point_sample_backward(gptr.data_ptr(), table.rows.data_ptr(),
                                                                    coords.data_ptr(), go.data_ptr(), table.R, K, stream))
        outs = [g.to(dt) if g is not None else None for g, (_, dt) in zip(grads, ctx.src_meta)]
        return (None, None, *outs)


def _backward_det(lib, table: _Rows, grads, coords, go, K, stream) -> None:
    """``msda_b200_point_sample_backward_det`` over the rows that need a gradient (the criterion's target rows need
    none, so compacting halves its sort)."""
    live, gptr, rows, key_base, keys = table.det_tables(grads)
    R = int(live.shape[0])
    if R == 0:
        return
    if R != table.R:
        go = go.index_select(0, torch.from_numpy(live).to(go.device, non_blocking=True))
    nbytes = lib.msda_b200_point_sample_backward_det_workspace_bytes(R, K, keys)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=go.device) if nbytes else None  # 0: the call reports why
    _cabi.check(lib.msda_b200_point_sample_backward_det(gptr.data_ptr(), rows.data_ptr(), key_base.data_ptr(), keys,
                                                        coords.data_ptr(), go.data_ptr(), R, K,
                                                        _cabi.ptr(ws), nbytes, stream))


def point_sample(sources: Sequence[torch.Tensor], src_id, plane_id, coords: torch.Tensor, coord_row) -> torch.Tensor:
    """Sample ``R`` planes at ``K`` points each; see the module docstring.

    ``sources``: CUDA tensors ``(n_j, h_j, w_j)``, float32 / bfloat16, or uint8 / bool for binary masks that need no
    gradient (non-contiguous ones are copied);
    ``src_id`` / ``plane_id`` / ``coord_row``: host integer arrays of length ``R``;
    ``coords``: ``(C, K, 2)`` CUDA float tensor of (x, y) in [0, 1]. Returns ``(R, K)`` float32.
    """
    if not isinstance(coords, torch.Tensor) or not coords.is_cuda:
        raise RuntimeError("point_sample: tensors must live on a CUDA device (this package has no CPU fallback)")
    if coords.dim() != 3 or coords.shape[-1] != 2:
        raise ValueError(f"point_sample: coords must be (C, K, 2), got {tuple(coords.shape)}")
    srcs = []
    for s in sources:
        if not s.is_cuda:
            raise RuntimeError("point_sample: tensors must live on a CUDA device (this package has no CPU fallback)")
        if s.dim() != 3:
            raise ValueError(f"point_sample: every source must be (n, h, w), got {tuple(s.shape)}")
        if s.dtype not in _DTYPE_CODE:
            raise TypeError(f"point_sample: float32, bfloat16, uint8 or bool sources only, got {s.dtype}")
        srcs.append(s if s.is_contiguous() else s.contiguous())
    coords = coords.detach().float().contiguous()
    table = _Rows(srcs, src_id, plane_id, coord_row, coords.device)
    if table.max_coord_row >= coords.shape[0]:
        raise ValueError("point_sample: coord_row out of range")
    return PointSampleFunction.apply(coords, table, *srcs)
