"""CPU-side checks of the drop-in boundary: the library loads and exports what the header declares."""
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


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "msda_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(msda_b200_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(lib):
    from weed_instance_segmentation_b200 import _cabi
    declared = _declared_symbols()
    assert declared, "no declarations parsed from include/msda_b200.h"
    assert sorted(_cabi.EXPORTS) == declared
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/msda_b200.h but not exported"


def test_abi_version_and_error_string(lib):
    from weed_instance_segmentation_b200 import _cabi
    assert lib.msda_b200_abi_version() == _cabi.ABI_VERSION
    assert lib.msda_b200_last_error() is not None


def test_desc_layout_matches_header_without_tile_schedule():
    from weed_instance_segmentation_b200 import _cabi
    text = open(os.path.join(ROOT, "include", "msda_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct msda_b200_desc \{(.*?)\} msda_b200_desc;", text, flags=re.S).group(1)
    members = re.findall(r"(\w+)\s*;", body)
    assert [name for name, _ in _cabi.Desc._fields_] == members
    # 10 x int32, two host pointers: 40 + 16 bytes on LP64
    assert ctypes.sizeof(_cabi.Desc) == 10 * 4 + 2 * ctypes.sizeof(ctypes.c_void_p)
    assert _cabi.Desc.spatial_shapes_hw.offset == 40
    assert _cabi.Desc.level_start_index.offset == 48


def test_validation_without_gpu(lib):
    """Argument validation happens before any CUDA call, so it is testable on the CPU box."""
    from weed_instance_segmentation_b200 import _cabi
    d, keep = _cabi.make_desc(1, 4, 2, 1, 32, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0])
    rc = lib.msda_b200_forward(d, None, None, None, None, None, None)
    assert rc == 1 and b"outside S" in lib.msda_b200_last_error()
    d, keep = _cabi.make_desc(1, 9, 2, 1, 24, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0])
    assert lib.msda_b200_forward(d, None, None, None, None, None, None) == 2  # unsupported head dim
    d, keep = _cabi.make_desc(1, 9, 2, 1, 32, 1, 1, _cabi.F32, _cabi.BF16, [(3, 3)], [0])
    assert lib.msda_b200_forward(d, None, None, None, None, None, None) == 2  # fp32 value + bf16 attn
    d, keep = _cabi.make_desc(1, 9, 2, 1, 32, 1, 1, _cabi.BF16, _cabi.BF16, [(3, 3)], [0])
    assert lib.msda_b200_backward_workspace_bytes(d) == 9 * 32 * 4
    d.flags = _cabi.FLAG_BF16_ATOMICS
    assert lib.msda_b200_backward_workspace_bytes(d) == 0
    # empty problems succeed without touching the device
    d, keep = _cabi.make_desc(0, 9, 2, 1, 32, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0])
    assert lib.msda_b200_forward(d, None, None, None, None, None, None) == 0


def test_no_cpu_fallback():
    import torch
    import weed_instance_segmentation_b200 as wis
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        wis.ms_deform_attn(torch.zeros(1, 4, 1, 16), [(2, 2)], None, torch.zeros(1, 2, 1, 1, 1, 2),
                           torch.zeros(1, 2, 1, 1, 1))


def test_product_never_imports_oracle():
    """The product package must not reference oracle/ (parity claims depend on it)."""
    pkg = os.path.join(ROOT, "weed_instance_segmentation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "msda_oracle" not in text, f


def test_new_entry_points_validate_before_touching_the_device(lib):
    """Host pipeline and point sampling: argument errors are reported without a GPU; empty work succeeds."""
    from weed_instance_segmentation_b200 import _cabi
    handle = ctypes.c_void_p()
    d, keep = _cabi.make_desc(2, 9, 9, 1, 32, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0])
    assert lib.msda_b200_host_pipeline_create(ctypes.byref(d), 1, 1, 1, None, ctypes.byref(handle)) == 1  # slots < 2
    assert b"slots" in lib.msda_b200_last_error() and not handle.value
    bad, keep2 = _cabi.make_desc(2, 9, 9, 1, 24, 1, 1, _cabi.F32, _cabi.F32, [(3, 3)], [0])
    assert lib.msda_b200_host_pipeline_create(ctypes.byref(bad), 1, 2, 1, None, ctypes.byref(handle)) == 2
    assert lib.msda_b200_host_pipeline_step(None, *([None] * 9)) == 1
    assert lib.msda_b200_host_pipeline_destroy(None) == 0
    assert lib.msda_b200_point_sample_forward(None, None, None, None, 0, 128, None) == 0   # no rows
    assert lib.msda_b200_point_sample_forward(None, None, None, None, 4, 128, None) == 1   # NULL tables
    assert lib.msda_b200_point_sample_backward(None, None, None, None, -1, 128, None) == 1
    assert ctypes.sizeof(ctypes.c_int32) * 4 == 16  # msda_b200_ps_row: four int32 (h, w, coord_row, dtype)
