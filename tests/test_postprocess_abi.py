"""CPU-side checks of the instance post-processing entry points in the C ABI: bad arguments are rejected before anything
touches a device, the workspace size is 0 for them, and the ABI version did not move."""
import ctypes

import pytest

NOT_NULL = ctypes.c_void_p(16)  # never dereferenced: the calls below fail or return before any device work
F32, BF16, U8 = 0, 1, 2


@pytest.fixture(scope="module")
def lib():
    from weed_instance_segmentation_b200 import build, _cabi
    build.build()
    return _cabi.load()


def _scores(lib, dtype=F32, C=3, B=2, Q=100, h=32, w=40, ptr=NOT_NULL, ws_bytes=1 << 30):
    return lib.msda_b200_postprocess_scores(ptr, dtype, ptr, C, ptr, B, Q, h, w, ptr, ptr, ws_bytes, None)


def _paint(lib, B=2, Q=100, max_h=384, ptr=NOT_NULL, ws_bytes=1 << 30):
    return lib.msda_b200_postprocess_paint(ptr, ws_bytes, ptr, ptr, 0.5, ptr, B, Q, max_h, ptr, ptr, None)


def _maps(lib, B=2, Q=100, image=0, H=200, W=300, n=3, ptr=NOT_NULL, ws_bytes=1 << 30):
    return lib.msda_b200_postprocess_binary_maps(ptr, ws_bytes, ptr, B, Q, image, H, W, n, ptr, None)


def test_abi_version_is_still_14(lib):
    from weed_instance_segmentation_b200 import _cabi
    assert lib.msda_b200_abi_version() == 14 == _cabi.ABI_VERSION


def test_workspace_bytes(lib):
    f = lib.msda_b200_postprocess_workspace_bytes
    assert f(2, 100, 3) == 2 * 100 * (384 * 384 // 8 + 4)
    assert f(1, 1, 1) == 384 * 384 // 8 + 4
    for B, Q, C in ((0, 100, 3), (-1, 100, 3), (2, 0, 3), (2, -5, 3), (2, 100, 0), (2, 100, -1),
                    (65536, 100, 3), (2, 1025, 3), (2, 1024, 2**21)):
        assert f(B, Q, C) == 0, (B, Q, C)


def test_scores_validates_before_touching_the_device(lib):
    for kw in (dict(B=0), dict(Q=-1), dict(C=0), dict(h=0), dict(w=-2)):
        assert _scores(lib, **kw) == 1, kw
        assert b"positive" in lib.msda_b200_last_error()
    for kw in (dict(B=65536), dict(Q=1025), dict(Q=1024, C=2**21)):
        assert _scores(lib, **kw) == 2, kw
    for dtype in (U8, 3, -1):
        assert _scores(lib, dtype=dtype) == 2
        assert b"F32 or BF16" in lib.msda_b200_last_error()
    assert _scores(lib, ptr=None) == 1
    assert b"NULL" in lib.msda_b200_last_error()
    assert _scores(lib, dtype=BF16, ws_bytes=2 * 100 * (18432 + 4) - 1) == 4
    assert b"workspace" in lib.msda_b200_last_error()


def test_paint_validates_before_touching_the_device(lib):
    for kw in (dict(B=0), dict(Q=0), dict(max_h=0), dict(max_h=-1)):
        assert _paint(lib, **kw) == 1, kw
        assert b"positive" in lib.msda_b200_last_error()
    assert _paint(lib, Q=1025) == 2
    assert _paint(lib, ptr=None) == 1
    assert b"NULL" in lib.msda_b200_last_error()
    assert _paint(lib, ws_bytes=0) == 4


def test_binary_maps_validates_before_touching_the_device(lib):
    for kw in (dict(B=0), dict(Q=-1)):
        assert _maps(lib, **kw) == 1, kw
    for kw in (dict(image=-1), dict(image=2), dict(H=0), dict(W=-1), dict(n=-1), dict(n=101)):
        assert _maps(lib, **kw) == 1, kw
        assert b"binary_maps" in lib.msda_b200_last_error()
    assert _maps(lib, ptr=None) == 1
    assert b"NULL" in lib.msda_b200_last_error()
    assert _maps(lib, ws_bytes=10) == 4
    # no instance: nothing to do, whatever the pointers
    assert _maps(lib, n=0, ptr=None) == 0


def test_python_entry_point_rejects_bad_inputs_without_a_device():
    import types

    import torch

    import weed_instance_segmentation_b200 as wis
    cpu = types.SimpleNamespace(class_queries_logits=torch.zeros(1, 4, 4), masks_queries_logits=torch.zeros(1, 4, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        wis.post_process_instance_segmentation(cpu)
    with pytest.raises(ValueError, match="can not be both"):
        wis.post_process_instance_segmentation(cpu, return_coco_annotation=True, return_binary_maps=True)
