"""Pixel-decoder input assembly on the B200 path (SURVEY.md section 8(f) rank 3).

Mirror of the assembly part of ``Mask2FormerPixelDecoder.forward`` (transformers 5.5.0,
``models/mask2former/modeling_mask2former.py:1287-1330`` = M2F:1287-1330), which the reference reaches from
``/root/reference/models/mask2former/train.py:196`` on every step:

* ``input_projections[level]`` = ``Conv2d(C_in, 256, 1)`` + ``GroupNorm(32, 256)``, then ``flatten(2).transpose(1, 2)``
  and ``torch.cat`` over the levels (M2F:1301-1313). Here the 1x1 convolution stays a library GEMM and ONE pair of
  kernels per level (``csrc/input_assembly.cu``) computes the GroupNorm statistics and writes the normalised,
  transposed rows straight into the concatenated ``(B, S, 256)`` encoder input -- no separate GroupNorm output, no
  concat copy; the backward is the matching pair.
* the sine position embedding (M2F:1304, :841-884): the reference rebuilds it for every level in every forward (its
  ``lru_cache(maxsize=1)`` is evicted by the next level) and for every batch item although it only depends on the
  level's shape. Here it is computed once per shape set with the reference's own module, for batch 1, and kept
  flattened and concatenated; per forward only ``level_embed`` is added (M2F:1315-1317). The result broadcasts over the
  batch where the reference materialises ``B`` copies.
* masks / ``valid_ratios`` / ``level_start_index`` (M2F:1306-1320) are constants of the shapes for un-padded inputs
  (all-False masks, ratios of one) and are cached.

``convert_pixel_decoder_inputs(model)`` rebinds ``forward`` of every ``Mask2FormerPixelDecoder`` inside ``model``; the
encoder call and the FPN tail (M2F:1322-1385) are the reference's code, restated below because ``forward`` cannot be
entered half way.
"""
from __future__ import annotations

import types

import torch
from torch import nn

from . import _cabi
from .functional import deterministic

_DTYPE_CODE = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}


class _GroupNormToRows(torch.autograd.Function):
    """``cat([GroupNorm(x_l).flatten(2).transpose(1, 2) for l], 1)`` for NCHW ``x_l`` -- float32 ``(B, S, C)``."""

    @staticmethod
    def forward(ctx, eps, groups, *tensors):
        lib = _cabi.load()
        L = len(tensors) // 3
        xs = [t.contiguous() for t in tensors[:L]]
        gammas = [t.detach().float().contiguous() for t in tensors[L:2 * L]]
        betas = [t.detach().float().contiguous() for t in tensors[2 * L:]]
        B, C = xs[0].shape[:2]
        hws = [x.shape[2] * x.shape[3] for x in xs]
        S = sum(hws)
        out = torch.empty((B, S, C), dtype=torch.float32, device=xs[0].device)
        stats = [torch.empty(B * groups * 2, dtype=torch.float32, device=out.device) for _ in xs]
        with torch.cuda.device(out.device):
            stream = torch.cuda.current_stream().cuda_stream
            start = 0
            for x, g, b, st, hw in zip(xs, gammas, betas, stats, hws):
                _cabi.check(lib.msda_b200_groupnorm_to_rows_forward(
                    x.data_ptr(), _DTYPE_CODE[x.dtype], g.data_ptr(), b.data_ptr(), float(eps),
                    out.data_ptr() + start * C * 4, S * C, st.data_ptr(), B, C, hw, groups, stream))
                start += hw
        ctx.save_for_backward(*xs, *gammas, *stats)
        ctx.meta = (L, groups, hws, [t.dtype for t in tensors[L:2 * L]], [t.dtype for t in tensors[2 * L:]])
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _cabi.load()
        L, groups, hws, gdt, bdt = ctx.meta
        saved = ctx.saved_tensors
        xs, gammas, stats = saved[:L], saved[L:2 * L], saved[2 * L:]
        grad_out = grad_out.float().contiguous()
        B, S, C = grad_out.shape
        gxs, ggs, gbs = [], [], []
        with torch.cuda.device(grad_out.device):
            stream = torch.cuda.current_stream().cuda_stream
            start = 0
            for x, g, st, hw in zip(xs, gammas, stats, hws):
                gx = torch.empty_like(x)
                gg = torch.zeros(C, dtype=torch.float32, device=x.device)
                gb = torch.zeros(C, dtype=torch.float32, device=x.device)
                scratch = torch.empty(B * groups * 2, dtype=torch.float32, device=x.device)
                _cabi.check(lib.msda_b200_groupnorm_to_rows_backward(
                    grad_out.data_ptr() + start * C * 4, S * C, x.data_ptr(), _DTYPE_CODE[x.dtype], g.data_ptr(),
                    st.data_ptr(), gx.data_ptr(), gg.data_ptr(), gb.data_ptr(), scratch.data_ptr(), B, C, hw, groups, stream))
                start += hw
                gxs.append(gx)
                ggs.append(gg)
                gbs.append(gb)
        return (None, None, *gxs, *[g.to(d) for g, d in zip(ggs, gdt)], *[b.to(d) for b, d in zip(gbs, bdt)])


def groupnorm_to_rows(xs, norms) -> torch.Tensor:
    """``xs``: the 1x1-conv outputs ``(B, C, H_l, W_l)`` (float32 / bfloat16, CUDA); ``norms``: their ``nn.GroupNorm``
    modules. Returns the concatenated, normalised, transposed ``(B, sum H_l*W_l, C)`` float32 tensor."""
    if not all(x.is_cuda for x in xs):
        raise RuntimeError("groupnorm_to_rows: tensors must live on a CUDA device (this package has no CPU fallback)")
    groups, eps = norms[0].num_groups, norms[0].eps
    if any(n.num_groups != groups or n.eps != eps or not n.affine for n in norms):
        raise ValueError("groupnorm_to_rows: the levels must share num_groups / eps and be affine")
    if any(x.dtype not in _DTYPE_CODE for x in xs):
        raise TypeError("groupnorm_to_rows: float32 or bfloat16 inputs")
    return _GroupNormToRows.apply(eps, groups, *xs, *[n.weight for n in norms], *[n.bias for n in norms])


class _Constants:
    """Shape-only constants of the assembly, built with the reference's own code for batch 1 / un-padded inputs."""

    def __init__(self):
        self.cache: dict = {}

    def get(self, decoder, shapes, batch, device, pos_dtype, embed_dtype):
        key = (tuple(shapes), batch, str(device), pos_dtype, embed_dtype)
        hit = self.cache.get(key)
        if hit is None:
            with torch.no_grad():
                c = decoder.level_embed.shape[1]
                sine = [decoder.position_embedding(torch.Size((1, c, h, w)), device, pos_dtype).flatten(2).transpose(1, 2)
                        for h, w in shapes]  # M2F:1304, :1314 -- the batch items are identical, one copy is kept
                sine = torch.cat(sine, 1).contiguous()  # (1, S, C)
                level_of_row = torch.cat([torch.full((h * w,), i, dtype=torch.long, device=device)
                                          for i, (h, w) in enumerate(shapes)])
                S = level_of_row.numel()
                sizes = torch.as_tensor(shapes, dtype=torch.long, device=device)
                hit = {
                    "sine": sine, "level_of_row": level_of_row,
                    "masks_flat": torch.zeros((batch, S), dtype=torch.bool, device=device),           # M2F:1306-1313
                    "level_start_index": torch.cat((sizes.new_zeros((1,)), sizes.prod(1).cumsum(0)[:-1])),  # M2F:1319
                    "valid_ratios": torch.ones((batch, len(shapes), 2), dtype=embed_dtype, device=device),  # M2F:1320
                }
            if len(self.cache) > 8:
                self.cache.clear()
            self.cache[key] = hit
        return hit


def assemble_encoder_inputs(decoder, features) -> dict:
    """Everything ``Mask2FormerPixelDecoder.forward`` hands to its encoder (M2F:1299-1320), from the backbone features."""
    if not hasattr(decoder, "_b200_constants"):
        decoder._b200_constants = _Constants()
    levels = features[::-1][: decoder.num_feature_levels]
    convs = [decoder.input_projections[i][0] for i in range(len(levels))]
    norms = [decoder.input_projections[i][1] for i in range(len(levels))]
    projected = [conv(x) for conv, x in zip(convs, levels)]  # the 1x1 convolutions: dense GEMMs, left to the library
    shapes = [(int(x.shape[2]), int(x.shape[3])) for x in projected]
    if deterministic():
        # the fused kernels accumulate grad_gamma / grad_beta with float atomics: the reference's own sequence instead
        embeds = torch.cat([norm(x).flatten(2).transpose(1, 2) for norm, x in zip(norms, projected)], 1)
    else:
        embeds = groupnorm_to_rows(projected, norms)
    const = decoder._b200_constants.get(decoder, shapes, embeds.shape[0], embeds.device, levels[0].dtype, embeds.dtype)
    # M2F:1315-1317: sine + level_embed[level]; (1, S, C), broadcasts over the batch
    pos = const["sine"] + decoder.level_embed.index_select(0, const["level_of_row"])[None].to(const["sine"].dtype)
    return {"inputs_embeds": embeds, "attention_mask": const["masks_flat"], "position_embeddings": pos,
            "spatial_shapes_list": shapes, "level_start_index": const["level_start_index"],
            "valid_ratios": const["valid_ratios"]}


class _ResizeBilinear(torch.autograd.Function):
    """``F.interpolate(x, size, mode="bilinear", align_corners=False)`` with a deterministic backward."""

    @staticmethod
    def forward(ctx, x, size):
        ctx.meta = (tuple(x.shape), x.dtype)
        # ATen's kernel itself: under the switch F.interpolate would take torch's decomposition instead, whose values
        # differ in the last bits from the kernel this backward is the adjoint of
        return torch.ops.aten.upsample_bilinear2d(x, list(size), False)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _cabi.load()
        (n, c, hi, wi), dtype = ctx.meta
        go = grad_out.float().contiguous()  # the kernel is fp32; other dtypes round-trip through it
        grad_in = torch.empty((n, c, hi, wi), dtype=torch.float32, device=go.device)
        with torch.cuda.device(go.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.msda_b200_resize_bilinear_backward(go.data_ptr() if go.numel() else None,
                                                               grad_in.data_ptr() if grad_in.numel() else None, n * c,
                                                               hi, wi, go.shape[2], go.shape[3], stream))
        return grad_in.to(dtype), None


def resize_bilinear(x: torch.Tensor, size) -> torch.Tensor:
    """``F.interpolate(x, size=size, mode="bilinear", align_corners=False)`` for an NCHW CUDA tensor, whose backward is
    ``csrc/resize_bilinear.cu``: a gather with one writer per input element, so the gradient is bit-identical run to run.
    torch's CUDA backward of the kernel scatters with atomics; under ``torch.use_deterministic_algorithms(True)``
    ``F.interpolate`` switches to a decomposition whose backward accumulates with ``index_put``, and whose forward values
    differ in the last bits from the switch-off path. Here the forward is the same kernel with the switch on or off."""
    if not x.is_cuda:
        raise RuntimeError("resize_bilinear: tensors must live on a CUDA device (this package has no CPU fallback)")
    if x.dim() != 4:
        raise ValueError(f"resize_bilinear: x must be (N, C, H, W), got {tuple(x.shape)}")
    return _ResizeBilinear.apply(x, tuple(int(v) for v in size))


def pixel_decoder_forward(self, features, encoder_outputs=None, output_attentions=None, output_hidden_states=None,
                          return_dict=None):
    """``Mask2FormerPixelDecoder.forward`` (M2F:1287-1385) with the input assembly above."""
    from transformers.models.mask2former.modeling_mask2former import Mask2FormerPixelDecoderOutput

    output_attentions = output_attentions if output_attentions is not None else self.config.output_attentions
    output_hidden_states = (output_hidden_states if output_hidden_states is not None
                            else self.config.output_hidden_states)
    enc_in = assemble_encoder_inputs(self, features)
    shapes = enc_in["spatial_shapes_list"]
    if encoder_outputs is None:  # M2F:1322-1334
        encoder_outputs = self.encoder(output_attentions=output_attentions, output_hidden_states=output_hidden_states,
                                       return_dict=return_dict, **enc_in)
    last_hidden_state = encoder_outputs.last_hidden_state
    batch_size = last_hidden_state.shape[0]
    # M2F:1339-1358: split the encoder output back into levels, NCHW
    sizes = [h * w for h, w in shapes]
    sizes[-1] = last_hidden_state.shape[1] - sum(sizes[:-1])
    outputs = [x.transpose(1, 2).view(batch_size, -1, h, w)
               for x, (h, w) in zip(torch.split(last_hidden_state, sizes, dim=1), shapes)]
    # M2F:1360-1371: extra FPN levels, low to high resolution
    for idx, feature in enumerate(features[: self.num_fpn_levels][::-1]):
        current_fpn = self.lateral_convolutions[idx](feature)
        if deterministic():  # a gather backward instead of torch's index_put-based one
            up = resize_bilinear(outputs[-1], current_fpn.shape[-2:])
        else:
            up = nn.functional.interpolate(outputs[-1], size=current_fpn.shape[-2:], mode="bilinear", align_corners=False)
        out = current_fpn + up
        outputs.append(self.output_convolutions[idx](out))
    multi_scale_features = tuple(outputs[: self.num_feature_levels])  # M2F:1373-1379
    return Mask2FormerPixelDecoderOutput(mask_features=self.mask_projection(outputs[-1]),
                                         multi_scale_features=multi_scale_features, attentions=encoder_outputs.attentions)


def convert_pixel_decoder_inputs(model: nn.Module) -> int:
    """Rebind ``forward`` of every ``Mask2FormerPixelDecoder`` in ``model`` to :func:`pixel_decoder_forward`
    (parameters and state-dict keys untouched). Only for un-padded batches, which is all the reference produces
    (``/root/reference/datasets/dataset_utils.py:45-53`` stacks equally sized images). Returns the number converted."""
    from transformers.models.mask2former import modeling_mask2former as m2f

    n = 0
    for module in model.modules():
        if isinstance(module, m2f.Mask2FormerPixelDecoder) and not getattr(module, "_b200_inputs", False):
            module.forward = types.MethodType(pixel_decoder_forward, module)
            module._b200_inputs = True
            n += 1
    return n
