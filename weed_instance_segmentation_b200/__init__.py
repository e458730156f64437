"""B200-native multi-scale deformable attention for the Mask2Former crop/weed model.

One hot path, hand-written for sm_100a behind a C ABI (``include/msda_b200.h``):
the pixel-decoder MSDeformAttn that ``marco-conciatori-public/weed_instance_segmentation``
runs through HuggingFace ``transformers`` (M2F:798-837). See DESIGN.md and INTEGRATION.md.
"""
from .functional import (  # noqa: F401
    MSDAError,
    MSDeformAttnFunction,
    ms_deform_attn,
    multi_scale_deformable_attention,
    query_order_2d,
)
from .fused import MSDeformAttnFusedFunction, ms_deform_attn_fused  # noqa: F401
from . import criterion  # noqa: F401
from .criterion import convert_criterion, restore_criterion  # noqa: F401
from .host import HostPipeline  # noqa: F401
from .pixel_decoder import convert_pixel_decoder_inputs, groupnorm_to_rows  # noqa: F401
from .point_sample import point_sample  # noqa: F401
from .hf_patch import install, installed, is_installed, uninstall  # noqa: F401
from .postprocess import post_process_instance_segmentation  # noqa: F401

__all__ = [
    "HostPipeline",
    "convert_pixel_decoder_inputs",
    "groupnorm_to_rows",
    "convert_criterion",
    "restore_criterion",
    "point_sample",
    "MSDAError",
    "MSDeformAttnFunction",
    "ms_deform_attn",
    "ms_deform_attn_fused",
    "multi_scale_deformable_attention",
    "query_order_2d",
    "install",
    "installed",
    "is_installed",
    "uninstall",
    "post_process_instance_segmentation",
]
