"""CPU-side checks of MSDA_B200_FLAG_DETERMINISTIC in the C ABI and its binding."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from weed_instance_segmentation_b200 import build, _cabi
    build.build()
    return _cabi.load()


def _header_define(name):
    text = open(os.path.join(ROOT, "include", "msda_b200.h")).read()
    return int(re.search(rf"#define {name} (\d+)u?\b", text).group(1))


def test_flag_matches_header_and_abi_version_is_14(lib):
    from weed_instance_segmentation_b200 import _cabi
    assert _header_define("MSDA_B200_FLAG_DETERMINISTIC") == _cabi.FLAG_DETERMINISTIC == 64
    assert _header_define("MSDA_B200_ABI_VERSION") == _cabi.ABI_VERSION == lib.msda_b200_abi_version() == 14
    others = [_cabi.FLAG_PROFILE, _cabi.FLAG_BWD_V1, _cabi.FLAG_STRICT_PADDING]
    assert all(f & _cabi.FLAG_DETERMINISTIC == 0 for f in others)
    assert _cabi.FLAG_DETERMINISTIC not in (2, 8, 32)  # the bits of the retired flags are not reused
    text = open(os.path.join(ROOT, "include", "msda_b200.h")).read()
    for retired in ("MSDA_B200_FLAG_BF16_ATOMICS", "MSDA_B200_FLAG_BWD_V2"):
        assert not re.search(rf"#define {retired}\b", text)


def test_deterministic_backward_validates_before_touching_the_device(lib):
    from weed_instance_segmentation_b200 import _cabi
    det = _cabi.FLAG_DETERMINISTIC
    null_args = [None] * 8 + [0, None, None]
    null_fused = [None] * 9 + [0, None, None]
    assert lib.msda_b200_backward(None, *null_args) == 1
    assert lib.msda_b200_backward_fused(None, *null_fused) == 1
    assert lib.msda_b200_backward_workspace_bytes(None) == 0
    cases = [
        ((1, 4, 2, 1, 32, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0]), 1, b"outside S"),
        ((1, 9, 2, 1, 24, 1, 1, _cabi.BF16, _cabi.BF16, [(3, 3)], [0]), 2, b"head dim"),
        ((1, 9, 2, 1, 32, 1, 1, _cabi.F32, _cabi.BF16, [(3, 3)], [0]), 2, b"fp32 values"),
        ((1, 9, 2, 1, 32, 1, 65, _cabi.BF16, _cabi.BF16, [(3, 3)], [0]), 2, b"L*P"),
    ]
    for args, code, msg in cases:
        d, keep = _cabi.make_desc(*args, flags=det)
        assert lib.msda_b200_backward(d, *null_args) == code
        assert msg in lib.msda_b200_last_error()
        assert lib.msda_b200_backward_fused(d, *null_fused) == code
        assert lib.msda_b200_backward_workspace_bytes(d) == 0
        handle = ctypes.c_void_p()
        assert lib.msda_b200_host_pipeline_create(ctypes.byref(d), 1, 2, 1, None, ctypes.byref(handle)) == code
        assert not handle.value
    # an empty batch succeeds without a device, whatever the tensor pointers (Q == S: implicit reference points)
    d, keep = _cabi.make_desc(0, 9, 9, 1, 32, 1, 1, _cabi.BF16, _cabi.BF16, [(3, 3)], [0], flags=det)
    assert lib.msda_b200_backward(d, *null_args) == 0
    assert lib.msda_b200_backward_fused(d, *null_fused) == 0


def test_deterministic_follows_the_torch_switch():
    import torch
    from weed_instance_segmentation_b200 import functional
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        assert functional.deterministic()
        torch.use_deterministic_algorithms(False)
        assert not functional.deterministic()
    finally:
        torch.use_deterministic_algorithms(prev)
