"""Host-side mirrors of the pixel-decoder modules that sit on the hot path.

* :class:`MSDeformAttn` mirrors ``Mask2FormerPixelDecoderEncoderMultiscaleDeformableAttention``
  (M2F:888-983): same parameter names (``sampling_offsets``, ``attention_weights``, ``value_proj``,
  ``output_proj``), same ``forward`` signature and return value, same ``ValueError`` on a bad
  ``reference_points`` last dim (M2F:978) and on ``embed_dim % num_heads`` (M2F:895-898).
* :class:`EncoderLayer` mirrors ``Mask2FormerPixelDecoderEncoderLayer`` (M2F:986-1072).
* :func:`convert_pixel_decoder` swaps both into a loaded HF model in place, re-using the
  existing ``nn.Parameter`` objects, so ``state_dict()`` keys, ``save_pretrained`` /
  ``from_pretrained`` (``/root/reference/models/mask2former/train.py:167-173,221-226``) and optimizer
  param groups are unchanged.

The dense projections stay on cuBLAS tensor cores (``F.linear``); everything between them --
bilinear gather, weighting, reduction over points and levels, and the gradient scatter -- runs in
``libmsda_b200.so``.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch import nn

from .functional import deterministic, ms_deform_attn
from .fused import ms_deform_attn_fused
from .layer_norm import add_layer_norm
from .linear import linear as _fused_linear
from .linear import linear_relu as _fused_linear_relu
from .linear import query_value_cast as _query_value_cast


class MSDeformAttn(nn.Module):
    """Multi-scale deformable attention module over the B200 operator."""

    def __init__(self, embed_dim: int, num_heads: int, n_levels: int, n_points: int):
        super().__init__()
        if embed_dim % num_heads != 0:
            raise ValueError(
                f"embed_dim (d_model) must be divisible by num_heads, but got {embed_dim} and {num_heads}"
            )
        self.d_model = embed_dim
        self.n_levels = n_levels
        self.n_heads = num_heads
        self.n_points = n_points
        self.im2col_step = 128  # kept for attribute compatibility (M2F:908); unused
        self.sampling_offsets = nn.Linear(embed_dim, num_heads * n_levels * n_points * 2)
        self.attention_weights = nn.Linear(embed_dim, num_heads * n_levels * n_points)
        self.value_proj = nn.Linear(embed_dim, embed_dim)
        self.output_proj = nn.Linear(embed_dim, embed_dim)
        # Mask2FormerPixelDecoder.forward always passes all-False padding masks (M2F:1307-1309), which
        # makes masked_fill (M2F:948-950) a full-tensor no-op; convert_pixel_decoder() sets this to skip it.
        self.assume_no_padding = False
        # Compute softmax and sampling locations inside the kernels (fused.py); convert_pixel_decoder() enables it.
        self.fused_prologue = False
        self.fused_linear = False  # projections with the fused bias-gradient reduction (linear.py)

    @classmethod
    def from_hf(cls, mod: nn.Module) -> "MSDeformAttn":
        """Wrap an HF module, sharing (not copying) its parameters."""
        new = cls.__new__(cls)
        nn.Module.__init__(new)
        new.d_model, new.n_levels, new.n_heads, new.n_points = mod.d_model, mod.n_levels, mod.n_heads, mod.n_points
        new.im2col_step = getattr(mod, "im2col_step", 128)
        new.sampling_offsets = mod.sampling_offsets
        new.attention_weights = mod.attention_weights
        new.value_proj = mod.value_proj
        new.output_proj = mod.output_proj
        new.assume_no_padding = False
        new.fused_prologue = False
        new.fused_linear = False
        new.implicit_reference_points = False
        new.train(mod.training)
        return new

    def _proj(self, layer: nn.Linear, x):
        """``layer(x)``; with ``fused_linear`` the bias gradient is reduced by the B200 column-sum kernel."""
        return _fused_linear(x, layer.weight, layer.bias) if self.fused_linear and not deterministic() else layer(x)

    @staticmethod
    def with_pos_embed(tensor, position_embeddings):
        return tensor if position_embeddings is None else tensor + position_embeddings

    def forward(
        self,
        hidden_states: torch.Tensor,
        attention_mask: torch.Tensor | None = None,
        encoder_hidden_states=None,
        encoder_attention_mask=None,
        position_embeddings: torch.Tensor | None = None,
        reference_points=None,
        spatial_shapes_list=None,
        level_start_index=None,
        output_attentions: bool = False,
    ):
        # Self-attention under bfloat16 autocast (the pixel decoder): the projections read bfloat16(hidden + pos) and
        # bfloat16(hidden) -- one kernel writes both (linear.query_value_cast) instead of an fp32 add and two casts.
        value_in = encoder_hidden_states
        if (self.fused_linear and position_embeddings is not None and encoder_hidden_states is hidden_states
                and hidden_states.is_cuda and hidden_states.dtype == torch.float32
                and position_embeddings.dtype == torch.float32 and position_embeddings.shape == hidden_states.shape
                and hidden_states.numel() % 8 == 0 and torch.is_autocast_enabled("cuda")
                and torch.get_autocast_dtype("cuda") == torch.bfloat16):
            hidden_states, value_in = _query_value_cast(hidden_states, position_embeddings)
        elif position_embeddings is not None:
            hidden_states = self.with_pos_embed(hidden_states, position_embeddings)
        batch_size, num_queries, _ = hidden_states.shape
        batch_size, sequence_length, _ = encoder_hidden_states.shape
        total_elements = sum(height * width for height, width in spatial_shapes_list)
        if total_elements != sequence_length:
            raise ValueError(
                "Make sure to align the spatial shapes with the sequence length of the encoder hidden states"
            )
        H, L, P = self.n_heads, self.n_levels, self.n_points

        if torch.is_autocast_enabled("cuda") and hidden_states.is_cuda and hidden_states.dtype == torch.float32:
            # both query projections read `hidden_states`: cast it to the autocast dtype ONCE (F.linear would do it twice)
            hidden_states = hidden_states.to(torch.get_autocast_dtype("cuda"))
        value = self._proj(self.value_proj, value_in)
        if attention_mask is not None and not self.assume_no_padding:
            value = value.masked_fill(attention_mask[..., None], float(0))
        value = value.view(batch_size, sequence_length, H, self.d_model // H)
        sampling_offsets = self._proj(self.sampling_offsets, hidden_states).view(batch_size, num_queries, H, L, P, 2)
        attention_weights = self._proj(self.attention_weights, hidden_states).view(batch_size, num_queries, H, L * P)
        if self.fused_prologue and reference_points.shape[-1] == 2 and not reference_points.requires_grad:
            # softmax (M2F:955-960) and ref + off / (W, H) (M2F:962-971) happen inside the kernels; in the pixel
            # decoder's self-attention (query i = pixel i, no padding) the reference points (M2F:1095-1125) do too
            implicit = self.implicit_reference_points and num_queries == sequence_length
            res = ms_deform_attn_fused(value, spatial_shapes_list, level_start_index, sampling_offsets,
                                       attention_weights, None if implicit else reference_points,
                                       return_attention_weights=output_attentions)
            output, attention_weights = res if output_attentions else (res, None)
            return self._proj(self.output_proj, output), attention_weights
        attention_weights = F.softmax(attention_weights, -1).view(batch_size, num_queries, H, L, P)
        if reference_points.shape[-1] == 2:
            offset_normalizer = torch.tensor(
                [[shape[1], shape[0]] for shape in spatial_shapes_list],
                dtype=reference_points.dtype, device=reference_points.device,
            )
            sampling_locations = (
                reference_points[:, :, None, :, None, :]
                + sampling_offsets / offset_normalizer[None, None, None, :, None, :]
            )
        elif reference_points.shape[-1] == 4:
            sampling_locations = (
                reference_points[:, :, None, :, None, :2]
                + sampling_offsets / P * reference_points[:, :, None, :, None, 2:] * 0.5
            )
        else:
            raise ValueError(f"Last dim of reference_points must be 2 or 4, but got {reference_points.shape[-1]}")

        output = ms_deform_attn(value, spatial_shapes_list, level_start_index, sampling_locations, attention_weights)
        output = self._proj(self.output_proj, output)
        return output, attention_weights


class EncoderLayer(nn.Module):
    """Pixel-decoder encoder layer: MSDeformAttn -> +res -> LN -> FFN -> +res -> LN (M2F:1005-1072)."""

    def __init__(self, embed_dim: int = 256, num_heads: int = 8, ffn_dim: int = 1024, dropout: float = 0.0,
                 n_levels: int = 3, n_points: int = 4):
        super().__init__()
        self.embed_dim = embed_dim
        self.self_attn = MSDeformAttn(embed_dim, num_heads, n_levels, n_points)
        self.self_attn_layer_norm = nn.LayerNorm(embed_dim)
        self.dropout = dropout
        self.activation_fn = F.relu
        self.activation_dropout = dropout
        self.fc1 = nn.Linear(embed_dim, ffn_dim)
        self.fc2 = nn.Linear(ffn_dim, embed_dim)
        self.final_layer_norm = nn.LayerNorm(embed_dim)
        self.fused_norm = False  # fused residual + LayerNorm kernels (layer_norm.py); convert_pixel_decoder() enables it
        self.fused_linear = False

    @classmethod
    def from_hf(cls, layer: nn.Module) -> "EncoderLayer":
        new = cls.__new__(cls)
        nn.Module.__init__(new)
        new.embed_dim = layer.embed_dim
        sa = layer.self_attn
        new.self_attn = sa if isinstance(sa, MSDeformAttn) else MSDeformAttn.from_hf(sa)
        new.self_attn_layer_norm = layer.self_attn_layer_norm
        new.dropout = layer.dropout
        new.activation_fn = layer.activation_fn
        new.activation_dropout = layer.activation_dropout
        new.fc1, new.fc2 = layer.fc1, layer.fc2
        new.final_layer_norm = layer.final_layer_norm
        new.fused_norm = False
        new.fused_linear = False
        new.train(layer.training)
        return new

    def _proj(self, layer: nn.Linear, x):
        return _fused_linear(x, layer.weight, layer.bias) if self.fused_linear and not deterministic() else layer(x)

    def _add_norm(self, branch, residual, norm, also_lowp=False, clamp=False):
        """``norm(residual + branch)`` (M2F:1049-1050, 1058-1059); one fused kernel when ``fused_norm`` is set.
        ``also_lowp``: return ``(y, y_bf16_or_None)`` -- the bfloat16 copy comes out of the same kernel.
        ``clamp``: also apply the layer's closing ``torch.clamp(y, -c, c)``, ``c = finfo(y.dtype).max - 1000``
        (M2F:1062-1065) -- inside the fused kernels when they run."""
        ok = (self.fused_norm and not deterministic() and branch.is_cuda and branch.shape[-1] % 128 == 0 and branch.shape[-1] <= 512
              and branch.dtype in (torch.float32, torch.bfloat16) and residual.dtype in (torch.float32, torch.bfloat16)
              and (torch.is_autocast_enabled() or (branch.dtype == residual.dtype == torch.float32)))
        if ok:
            lowp = also_lowp and torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16
            c = float(torch.finfo(torch.float32).max - 1000) if clamp else None  # the fused kernels return float32
            res = add_layer_norm(branch, residual, norm.weight, norm.bias, norm.eps, also_lowp=lowp, clamp=c)
            return (res if lowp else (res, None)) if also_lowp else res
        y = norm(residual + branch)
        if clamp:
            c = torch.finfo(y.dtype).max - 1000
            y = torch.clamp(y, min=-c, max=c)
        return (y, None) if also_lowp else y

    def forward(
        self,
        hidden_states: torch.Tensor,
        attention_mask: torch.Tensor,
        position_embeddings: torch.Tensor | None = None,
        reference_points=None,
        spatial_shapes_list=None,
        level_start_index=None,
        output_attentions: bool = False,
    ):
        residual = hidden_states
        hidden_states, attn_weights = self.self_attn(
            hidden_states=hidden_states,
            attention_mask=attention_mask,
            encoder_hidden_states=hidden_states,
            encoder_attention_mask=attention_mask,
            position_embeddings=position_embeddings,
            reference_points=reference_points,
            spatial_shapes_list=spatial_shapes_list,
            level_start_index=level_start_index,
            output_attentions=output_attentions,
        )
        hidden_states = F.dropout(hidden_states, p=self.dropout, training=self.training)
        # the first LayerNorm also emits its output in bfloat16 (under autocast): fc1 reads that copy, no cast kernel
        hidden_states, lowp = self._add_norm(hidden_states, residual, self.self_attn_layer_norm, also_lowp=True)

        residual = hidden_states
        fc1_in = lowp if lowp is not None else hidden_states
        if self.fused_linear and self.activation_fn is F.relu and not deterministic():
            hidden_states = _fused_linear_relu(fc1_in, self.fc1.weight, self.fc1.bias)  # bias + ReLU in the GEMM epilogue
        else:
            hidden_states = self.activation_fn(self._proj(self.fc1, fc1_in))
        hidden_states = F.dropout(hidden_states, p=self.activation_dropout, training=self.training)
        hidden_states = self._proj(self.fc2, hidden_states)
        hidden_states = F.dropout(hidden_states, p=self.dropout, training=self.training)
        # The reference clamps only `if not torch.isfinite(hidden_states).all()` (M2F:1062-1065), a device->host sync
        # per layer per step. The clamp bounds are finfo.max - 1000, so for finite inputs it is the identity and NaN
        # passes through unchanged: applying it unconditionally gives the same tensor without stalling the stream, and
        # the fused LayerNorm kernels apply it (and its backward mask) in place of five elementwise kernels.
        hidden_states = self._add_norm(hidden_states, residual, self.final_layer_norm, clamp=self.training)

        outputs = (hidden_states,)
        if output_attentions:
            outputs += (attn_weights.transpose(1, 0),)
        return outputs


def _cached_reference_points(original):
    """``get_reference_points`` (M2F:1095-1125) for un-padded inputs: ``valid_ratios`` is all ones, so the result is a
    constant of (shapes, batch, device, dtype) -- computed once with the reference's own code, then reused (the
    reference rebuilds it, ~20 small kernels, in every forward). The fused kernels do not even read it
    (``implicit_reference_points``); HF's encoder loop still passes it along."""
    cache: dict = {}

    def get_reference_points(spatial_shapes_list, valid_ratios, device):
        key = (tuple(tuple(s) for s in spatial_shapes_list), tuple(valid_ratios.shape), str(device), valid_ratios.dtype)
        hit = cache.get(key)
        if hit is None:
            hit = original(spatial_shapes_list, torch.ones_like(valid_ratios), device).detach()
            if len(cache) > 16:
                cache.clear()
            cache[key] = hit
        return hit

    get_reference_points._b200_cache = cache
    return get_reference_points


def convert_pixel_decoder(model: nn.Module, assume_no_padding: bool = True, fused_prologue: bool = True,
                          fused_norm: bool = True, fused_linear: bool = True) -> int:
    """Replace every HF pixel-decoder encoder layer (and its MSDeformAttn) inside ``model`` by the
    mirrors above, sharing parameters. Returns the number of layers converted.

    ``model`` is what ``/root/reference/models/model_utils.py:13-14`` returns
    (``Mask2FormerForUniversalSegmentation``) or any sub-module of it.
    """
    from transformers.models.mask2former import modeling_mask2former as m2f

    converted = 0
    for module in model.modules():
        if isinstance(module, m2f.Mask2FormerPixelDecoderEncoderOnly):
            if assume_no_padding and not hasattr(module.get_reference_points, "_b200_cache"):
                module.get_reference_points = _cached_reference_points(module.get_reference_points)
            for i, layer in enumerate(module.layers):
                if isinstance(layer, EncoderLayer):
                    continue
                new = EncoderLayer.from_hf(layer)
                new.self_attn.assume_no_padding = assume_no_padding
                new.self_attn.implicit_reference_points = assume_no_padding and fused_prologue
                new.self_attn.fused_prologue = fused_prologue
                new.fused_norm = fused_norm
                new.fused_linear = new.self_attn.fused_linear = fused_linear
                module.layers[i] = new
                converted += 1
    return converted
