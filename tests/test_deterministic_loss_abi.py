"""CPU-side checks of the deterministic point-sampling and bilinear-resize backwards in the C ABI: bad arguments are
rejected before anything touches a device, and empty work succeeds without one."""
import ctypes

import pytest

NOT_NULL = ctypes.c_void_p(16)  # never dereferenced: the calls below fail or return before any device work


@pytest.fixture(scope="module")
def lib():
    from weed_instance_segmentation_b200 import build, _cabi
    build.build()
    return _cabi.load()


def _ps_det(lib, R, K, keys, tables=NOT_NULL):
    return lib.msda_b200_point_sample_backward_det(tables, tables, tables, keys, tables, tables, R, K, None, 0, None)


def test_point_sample_backward_det_validates_before_touching_the_device(lib):
    for R, K, keys in ((-1, 4, 10), (2, -1, 10), (2, 4, -1)):
        assert _ps_det(lib, R, K, keys) == 1
        assert b"negative" in lib.msda_b200_last_error()
        assert lib.msda_b200_point_sample_backward_det_workspace_bytes(R, K, keys) == 0
    assert _ps_det(lib, 2, 4, 10, tables=None) == 1
    assert b"NULL" in lib.msda_b200_last_error()
    # unsupported: the sort key needs 32 bits for the sentinel, the record index 31
    assert _ps_det(lib, 2, 4, 2**32 - 1) == 2
    assert b"2^32 - 1" in lib.msda_b200_last_error()
    assert lib.msda_b200_point_sample_backward_det_workspace_bytes(2, 4, 2**32 - 1) == 0
    for R, K in ((2**29, 1), (2**20, 2**9), (2**31 - 1, 2**31 - 1)):
        assert _ps_det(lib, R, K, 10) == 2
        assert b"records" in lib.msda_b200_last_error()
        assert lib.msda_b200_point_sample_backward_det_workspace_bytes(R, K, 10) == 0
    # empty work: nothing to do, whatever the pointers
    for R, K in ((0, 4), (2, 0), (0, 0)):
        assert _ps_det(lib, R, K, 0, tables=None) == 0
        assert lib.msda_b200_point_sample_backward_det_workspace_bytes(R, K, 0) == 0


def test_resize_bilinear_backward_validates_before_touching_the_device(lib):
    f = lib.msda_b200_resize_bilinear_backward
    for nc, hi, wi, ho, wo in ((-1, 2, 2, 4, 4), (1, 0, 2, 4, 4), (1, 2, -3, 4, 4), (1, 2, 2, 0, 4), (1, 2, 2, 4, -1)):
        assert f(NOT_NULL, NOT_NULL, nc, hi, wi, ho, wo, None) == 1
        assert b"resize_bilinear" in lib.msda_b200_last_error()
    assert f(None, NOT_NULL, 1, 2, 2, 4, 4, None) == 1
    assert f(NOT_NULL, None, 1, 2, 2, 4, 4, None) == 1
    assert b"NULL" in lib.msda_b200_last_error()
    assert f(NOT_NULL, NOT_NULL, 2**40, 2**15, 2**15, 4, 4, None) == 2
    assert f(None, None, 0, 121, 162, 242, 324, None) == 0
