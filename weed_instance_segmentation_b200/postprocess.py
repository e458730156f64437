"""Instance post-processing of Mask2Former outputs on the device.

``post_process_instance_segmentation`` returns what ``Mask2FormerImageProcessor.post_process_instance_segmentation``
(transformers 5.5.0, ``image_processing_mask2former.py:605-724``, "M2FIP") returns, with M2FIP's quirks:
``mask_threshold`` and ``overlap_mask_area_threshold`` are ignored, masks are ``logit > 0`` on the 384 x 384 resampling,
a selection is kept when its mask is non-empty *after* the nearest resize to the target size and its score reaches
``threshold``, one query may be selected under two labels, and later kept selections overwrite earlier ones.

M2FIP synchronises with the device at least twice per selection and copies every kept mask to the host. Here the class
side runs M2FIP's own torch calls, the mask side runs two batched kernels (``csrc/postprocess.cu``), and one copy from a
pinned buffer brings back the maps and the (score, label, id) table of the whole batch.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _cabi
from ._cabi import DTYPE_CODE


def post_process_instance_segmentation(outputs, threshold: float = 0.5, mask_threshold: float = 0.5,
                                       overlap_mask_area_threshold: float = 0.8, target_sizes=None,
                                       return_coco_annotation: bool | None = False,
                                       return_binary_maps: bool | None = False) -> list[dict]:
    """M2FIP's instance post-processing of ``outputs`` (``class_queries_logits`` (B, Q, C+1) and
    ``masks_queries_logits`` (B, Q, h, w), float32 or bfloat16, on a CUDA device).

    Returns one ``{"segmentation", "segments_info"}`` dict per image: ``segmentation`` is a host float32 (H, W) map of
    segment ids with -1 for background, its COCO run-length encoding with ``return_coco_annotation``, or the
    (n_instances, H, W) float32 device tensor of binary maps with ``return_binary_maps`` (when there is an instance);
    ``segments_info`` lists ``{"id", "label_id", "was_fused": False, "score"}`` in selection order.
    ``mask_threshold`` and ``overlap_mask_area_threshold`` are accepted and ignored, as in M2FIP.
    """
    if return_coco_annotation and return_binary_maps:
        raise ValueError("return_coco_annotation and return_binary_maps can not be both set to True.")
    cls = outputs.class_queries_logits
    masks = outputs.masks_queries_logits
    if not (cls.is_cuda and masks.is_cuda) or cls.device != masks.device:
        raise RuntimeError("post_process_instance_segmentation: outputs must live on one CUDA device "
                           "(this package has no CPU fallback)")
    for name, t in (("class_queries_logits", cls), ("masks_queries_logits", masks)):
        if t.dtype not in DTYPE_CODE:
            raise TypeError(f"post_process_instance_segmentation: {name} has dtype {t.dtype}; float32 or bfloat16 only")
    if cls.dim() != 3 or masks.dim() != 4 or masks.shape[:2] != cls.shape[:2] or cls.shape[-1] < 2:
        raise ValueError(f"post_process_instance_segmentation: class logits {tuple(cls.shape)} (B, Q, C+1 >= 2) and "
                         f"mask logits {tuple(masks.shape)} (B, Q, h, w) do not match")
    B, Q = cls.shape[:2]
    C = cls.shape[-1] - 1
    if target_sizes is None:
        sizes = [(384, 384)] * B  # the nearest resize from 384 x 384 to 384 x 384 is the identity
    else:
        if len(target_sizes) != B:
            raise ValueError(f"post_process_instance_segmentation: {len(target_sizes)} target sizes for {B} images")
        sizes = [(int(h), int(w)) for h, w in target_sizes]
        if any(h <= 0 or w <= 0 for h, w in sizes):
            raise ValueError(f"post_process_instance_segmentation: target sizes must be positive, got {sizes}")
    lib = _cabi.load()
    dev = masks.device
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        # Class side: M2FIP's own calls, image by image, so the selection order is its own.
        top_scores, top_index = [], []
        for i in range(B):
            scores = torch.nn.functional.softmax(cls[i], dim=-1)[:, :-1]
            s, k = scores.flatten(0, 1).topk(Q, sorted=False)
            top_scores.append(s)
            top_index.append(k)
        scores_per_image = torch.stack(top_scores)
        topk_index = torch.stack(top_index)
        labels = torch.arange(C, device=dev).unsqueeze(0).repeat(Q, 1).flatten(0, 1)[topk_index]
        hw = torch.tensor(sizes, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)
        masks = masks.contiguous()
        ws_bytes = lib.msda_b200_postprocess_workspace_bytes(B, Q, C)
        if ws_bytes == 0:
            raise ValueError(f"post_process_instance_segmentation: unsupported B={B}, Q={Q}, C={C} "
                             "(B <= 65535, Q <= 1024, Q*C < 2^31)")
        workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        mask_score = torch.empty((B, Q), dtype=torch.float32, device=dev)
        _cabi.check(lib.msda_b200_postprocess_scores(
            masks.data_ptr(), DTYPE_CODE[masks.dtype], topk_index.data_ptr(), C, hw.data_ptr(), B, Q, masks.shape[2],
            masks.shape[3], mask_score.data_ptr(), workspace.data_ptr(), ws_bytes, stream))
        pred_scores = (scores_per_image * mask_score).contiguous()  # float32 for either class-logit dtype
        n_map = sum(h * w for h, w in sizes)
        out = torch.empty(n_map + 3 * B * Q, dtype=torch.float32, device=dev)  # maps, then the (score, label, id) table
        table = out[n_map:].view(torch.int32)
        _cabi.check(lib.msda_b200_postprocess_paint(
            workspace.data_ptr(), ws_bytes, pred_scores.data_ptr(), labels.data_ptr(), float(threshold), hw.data_ptr(),
            B, Q, max(h for h, _ in sizes), out.data_ptr(), table.data_ptr(), stream))
        host = torch.empty(out.shape, dtype=torch.float32, pin_memory=True)
        host.copy_(out)  # the call's one device-to-host transfer; it waits for the kernels
        host_table = host.numpy()[n_map:].reshape(B, Q, 3)
        host_scores = host_table[:, :, 0]
        host_table = host_table.view(np.int32)

        if return_coco_annotation:
            from transformers.models.mask2former.image_processing_mask2former import convert_segmentation_to_rle
        results, off = [], 0
        for i, (h, w) in enumerate(sizes):
            # a pageable copy: the pinned staging buffer goes back to torch's host cache for the next call instead
            # of staying page-locked for as long as the caller keeps the results
            segmentation = host[off:off + h * w].view(h, w).clone()
            off += h * w
            kept = np.flatnonzero(host_table[i, :, 2] >= 0)
            segments = [{"id": int(host_table[i, j, 2]), "label_id": int(host_table[i, j, 1]), "was_fused": False,
                         "score": round(float(host_scores[i, j]), 6)} for j in kept]
            if return_coco_annotation:
                segmentation = convert_segmentation_to_rle(segmentation)
            if return_binary_maps and len(segments) != 0:
                segmentation = torch.empty((len(segments), h, w), dtype=torch.float32, device=dev)
                _cabi.check(lib.msda_b200_postprocess_binary_maps(
                    workspace.data_ptr(), ws_bytes, table.data_ptr(), B, Q, i, h, w, len(segments),
                    segmentation.data_ptr(), stream))
            results.append({"segmentation": segmentation, "segments_info": segments})
    return results
