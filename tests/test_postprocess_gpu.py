"""Instance post-processing on the device vs Mask2FormerImageProcessor.post_process_instance_segmentation (transformers
5.5.0, image_processing_mask2former.py:605-724, "M2FIP") run on the same device and inputs."""
import itertools
import types
import warnings

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SIZE = 384
SMALL, LARGE = (200, 300), (966, 1296)


@pytest.fixture(scope="module")
def m2fip():
    pytest.importorskip("transformers")
    from transformers import Mask2FormerImageProcessor
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()
    _cabi.load()
    return Mask2FormerImageProcessor().post_process_instance_segmentation


def _outputs(cls, masks):
    return types.SimpleNamespace(class_queries_logits=cls, masks_queries_logits=masks)


def _all_scores(cls, masks):
    """pred_scores of every selection, computed with M2FIP's arithmetic (the threshold-gap check needs them all)."""
    up = F.interpolate(masks, size=(SIZE, SIZE), mode="bilinear", align_corners=False)
    B, Q, C = cls.shape[0], cls.shape[1], cls.shape[2] - 1
    out = []
    for i in range(B):
        s, k = F.softmax(cls[i], dim=-1)[:, :-1].flatten(0, 1).topk(Q, sorted=False)
        m = up[i][torch.div(k, C, rounding_mode="floor")]
        pm = (m > 0).float()
        out.append(s * (m.sigmoid().flatten(1) * pm.flatten(1)).sum(1) / (pm.flatten(1).sum(1) + 1e-6))
    return torch.stack(out)


def _inputs(dtype, B, C, hw, thresholds, seed, Q=100):
    """Random class and mask logits whose selection scores all keep 1e-5 away from every positive threshold (a score is
    never negative, so the comparison with 0.0 cannot flip)."""
    for s in range(seed, seed + 50):
        g = torch.Generator(device="cuda").manual_seed(s)
        cls = 2 * torch.randn(B, Q, C + 1, generator=g, device="cuda")
        # one confident class for a random share of the queries, so that scores spread over (0, 1)
        boost = 10 * torch.rand(B, Q, 1, generator=g, device="cuda")
        pick = torch.randint(0, C + 1, (B, Q, 1), generator=g, device="cuda")
        cls.scatter_add_(2, pick, boost)
        masks = torch.randn(B, Q, *hw, generator=g, device="cuda") + 0.3 * torch.randn(B, Q, 1, 1, generator=g,
                                                                                       device="cuda")
        cls, masks = cls.to(dtype), masks.to(dtype)
        scores = _all_scores(cls, masks)
        if all(float((scores - t).abs().min()) > 1e-5 for t in thresholds if t > 0):
            return cls, masks
    raise AssertionError("no seed kept every score away from the thresholds")


def _ambiguous(masks_i, tol, shape):
    """Pixels of a target-size map that may change owner: some query's 384^2 upsampled logit lies within tol of 0
    (the rule of test_model_gpu.py::test_instance_masks_unchanged), carried to the target size as M2FIP does."""
    up = F.interpolate(masks_i[None], size=(SIZE, SIZE), mode="bilinear", align_corners=False)[0]
    amb = (up.float().abs() < tol).any(0).float()[None, None]
    return F.interpolate(amb, size=tuple(shape), mode="nearest")[0, 0].cpu() > 0


def _compare(ref, got, masks, binary=False):
    """segments_info entry for entry; maps equal outside the ambiguous pixels. Returns the differing-pixel count."""
    tol = 1e-4 * masks.float().abs().max().item()
    differing = 0
    assert len(ref) == len(got)
    for i, (a, b) in enumerate(zip(ref, got)):
        assert len(a["segments_info"]) == len(b["segments_info"]), i
        for sa, sb in zip(a["segments_info"], b["segments_info"]):
            assert (sa["id"], sa["label_id"], sa["was_fused"]) == (sb["id"], sb["label_id"], sb["was_fused"])
            assert abs(sa["score"] - sb["score"]) <= 2e-6, (sa, sb)
        ma, mb = a["segmentation"], b["segmentation"]
        assert ma.shape == mb.shape and ma.dtype == mb.dtype == torch.float32
        if binary and a["segments_info"]:
            assert ma.is_cuda and mb.is_cuda
        else:
            assert not mb.is_cuda
        diff = (ma.cpu() != mb.cpu())
        if diff.any():
            amb = _ambiguous(masks[i], tol, ma.shape[-2:])
            assert not (diff & ~amb).any(), f"image {i}: {int((diff & ~amb).sum())} unexplained differing pixels"
        differing += int(diff.sum())
    return differing


def _targets(kind, B):
    return {"none": None, "small": [SMALL] * B, "large": [LARGE] * B,
            "mixed": [(SMALL, LARGE, (384, 384))[i % 3] for i in range(B)]}[kind]


CASES = [(dtype, hw, kind, (1, 3)[n % 2], (3, 80)[(n // 2) % 2])
         for n, (dtype, hw, kind) in enumerate(itertools.product(
             (torch.float32, torch.bfloat16), ((32, 40), (242, 324), (512, 512)), ("none", "small", "large", "mixed")))]


@pytest.mark.parametrize("dtype,hw,kind,B,C", CASES,
                         ids=[f"{str(d)[6:]}-{h}x{w}-{k}-B{b}-C{c}" for d, (h, w), k, b, c in CASES])
def test_random_logits_match_m2fip(m2fip, dtype, hw, kind, B, C):
    import weed_instance_segmentation_b200 as wis
    thresholds = (0.0, 0.5, 0.9)
    cls, masks = _inputs(dtype, B, C, hw, thresholds, seed=100 * CASES.index((dtype, hw, kind, B, C)))
    target_sizes = _targets(kind, B)
    differing, kept = 0, 0
    for t in thresholds:
        ref = m2fip(_outputs(cls, masks), threshold=t, target_sizes=target_sizes)
        got = wis.post_process_instance_segmentation(_outputs(cls, masks), threshold=t, target_sizes=target_sizes)
        differing += _compare(ref, got, masks)
        kept += sum(len(r["segments_info"]) for r in ref)
    assert kept > 0
    print(f"differing pixels (all ambiguous): {differing}")


def test_planted_cases(m2fip):
    """An all-negative query; a mask set only at 384^2 pixel (1, 1), which the nearest resize to 100 x 100 never samples;
    one query selected under two labels; two overlapping masks, where the later selection owns the overlap."""
    import weed_instance_segmentation_b200 as wis
    Q, C = 10, 3
    masks = torch.full((1, Q, SIZE, SIZE), -5.0, device="cuda")  # 384^2 planes: the bilinear resize is the identity
    cls = torch.full((1, Q, C + 1), -10.0, device="cuda")
    cls[0, 0, 0] = 10.0                                            # q0: confident class, all-negative mask
    masks[0, 1, 1, 1] = 5.0                                        # q1: one pixel, on no sampled row of a 100 x 100 map
    cls[0, 1, 1] = 10.0
    masks[0, 2, 50:150, 50:150] = 5.0                              # q2: two labels at about 0.5 each
    cls[0, 2, 0] = cls[0, 2, 2] = 10.0
    masks[0, 3, 100:200, 100:200] = 5.0                            # q3: overlaps q2
    cls[0, 3, 1] = 10.0
    out = _outputs(cls, masks)
    for target_sizes in ([(100, 100)], None):
        ref = m2fip(out, threshold=0.3, target_sizes=target_sizes)
        got = wis.post_process_instance_segmentation(out, threshold=0.3, target_sizes=target_sizes)
        assert _compare(ref, got, masks) == 0
        seg, info = got[0]["segmentation"], got[0]["segments_info"]
        # q2 twice (labels 0 and 2) and q3; q1 only where its pixel survives; never q0
        labels = sorted(s["label_id"] for s in info)
        assert labels == ([0, 1, 2] if target_sizes else [0, 1, 1, 2]), info
        # q2's first selection is entirely overwritten by its second one
        present = set(int(v) for v in seg.unique().tolist() if v >= 0)
        assert len(present) == len(info) - 1
        ids_q2 = [s["id"] for s in info if s["label_id"] in (0, 2)]
        id_q3 = [s["id"] for s in info if s["label_id"] == 1 and s["id"] in present and
                 (seg == s["id"]).sum() > 100][0]
        sy = 100 / SIZE if target_sizes else 1.0
        y0, y1 = int(110 * sy), int(140 * sy)  # inside the overlap [100, 150)^2
        assert (seg[y0:y1, y0:y1] == max(max(ids_q2), id_q3)).all()


def test_binary_maps_and_coco_annotation_match_m2fip(m2fip):
    from transformers.models.mask2former.image_processing_mask2former import convert_segmentation_to_rle

    import weed_instance_segmentation_b200 as wis
    cls, masks = _inputs(torch.float32, 2, 3, (242, 324), (0.5,), seed=7)
    out = _outputs(cls, masks)
    for kw in (dict(threshold=0.5, target_sizes=[SMALL, LARGE]), dict(threshold=0.5, target_sizes=None)):
        ref = m2fip(out, return_binary_maps=True, **kw)
        got = wis.post_process_instance_segmentation(out, return_binary_maps=True, **kw)
        assert any(r["segments_info"] for r in ref)
        _compare(ref, got, masks, binary=True)
        plain_ref, plain = m2fip(out, **kw), wis.post_process_instance_segmentation(out, **kw)
        ref = m2fip(out, return_coco_annotation=True, **kw)
        got = wis.post_process_instance_segmentation(out, return_coco_annotation=True, **kw)
        for a, b, pa, pb in zip(ref, got, plain_ref, plain):
            assert b["segmentation"] == convert_segmentation_to_rle(pb["segmentation"])
            if pa["segmentation"].equal(pb["segmentation"]):  # else they differ at ambiguous pixels (_compare above)
                assert a["segmentation"] == b["segmentation"]


def test_converted_model_instances_match(m2fip):
    """A random-init converted model at the config-1 shape (batch 1, 512 x 512, fp32) gives the same instances through
    M2FIP and the device post-processing."""
    import weed_instance_segmentation_b200 as wis
    from weed_instance_segmentation_b200 import train
    model = train.build_model("swin_tiny_test", num_labels=3, seed=0).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(0)
    pixel_values = torch.randn(1, 3, 512, 512, generator=g, device="cuda")
    with torch.no_grad(), wis.installed():
        out = model(pixel_values=pixel_values)
    # threshold 0.0: every non-empty selection is kept, and no score can sit on the wrong side of it
    kw = dict(threshold=0.0, target_sizes=[(512, 512)])
    ref, got = m2fip(out, **kw), wis.post_process_instance_segmentation(out, **kw)
    assert ref[0]["segments_info"]
    print(f"{len(ref[0]['segments_info'])} instances, differing pixels (all ambiguous): "
          f"{_compare(ref, got, out.masks_queries_logits)}")


def test_repeat_and_side_stream_are_byte_identical(m2fip):
    import weed_instance_segmentation_b200 as wis
    cls, masks = _inputs(torch.bfloat16, 3, 80, (242, 324), (0.0,), seed=3)
    kw = dict(threshold=0.0, target_sizes=[SMALL, LARGE, (384, 384)], return_binary_maps=True)
    runs = [wis.post_process_instance_segmentation(_outputs(cls, masks), **kw) for _ in range(2)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        runs.append(wis.post_process_instance_segmentation(_outputs(cls, masks), **kw))
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for other in runs[1:]:
        for a, b in zip(runs[0], other):
            assert a["segments_info"] == b["segments_info"]
            assert a["segmentation"].cpu().view(torch.int32).equal(b["segmentation"].cpu().view(torch.int32))


def _sync_count(fn):
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            fn()
        finally:
            torch.cuda.set_sync_debug_mode(0)
    # only the per-operation warnings; setting the mode also emits a one-time "prototype feature" notice
    return sum("called a synchronizing CUDA operation" in str(w.message) for w in caught)


def test_one_synchronisation_per_call(m2fip):
    import weed_instance_segmentation_b200 as wis
    cls, masks = _inputs(torch.float32, 2, 3, (242, 324), (0.5,), seed=11)
    kw = dict(threshold=0.5, target_sizes=[SMALL, LARGE])
    wis.post_process_instance_segmentation(_outputs(cls, masks), **kw)  # warm-up: library load, pinned-memory pool
    torch.cuda.synchronize()
    ours = _sync_count(lambda: wis.post_process_instance_segmentation(_outputs(cls, masks), **kw))
    theirs = _sync_count(lambda: m2fip(_outputs(cls, masks), **kw))
    print(f"synchronising operations per call: {ours} vs M2FIP {theirs}")
    assert ours == 1
    assert theirs >= 2 * 100 * 2


def test_input_errors(m2fip):
    import weed_instance_segmentation_b200 as wis
    cls = torch.zeros(2, 5, 4, device="cuda")
    masks = torch.zeros(2, 5, 8, 8, device="cuda")
    with pytest.raises(TypeError):
        wis.post_process_instance_segmentation(_outputs(cls.half(), masks))
    with pytest.raises(TypeError):
        wis.post_process_instance_segmentation(_outputs(cls, masks.double()))
    with pytest.raises(ValueError):
        wis.post_process_instance_segmentation(_outputs(cls, masks), target_sizes=[(10, 10)])
    with pytest.raises(RuntimeError):
        wis.post_process_instance_segmentation(_outputs(cls.cpu(), masks))
