"""Images of any numeric element type, the parts that need no GPU: the _px entry points' argument
errors (codes + messages, nothing touches a device) and the dtype table of the engine."""

import ctypes
import re

import numpy as np
import pytest

from photonbend_b200 import _native, engine

FAKE = ctypes.c_void_p(256)  # never dereferenced: validation fails first


def _src_desc(kind):
    d = _native.ImageDesc()
    d.kind, d.height, d.width = kind, 8, 16
    d.lens, d.fov, d.f_distance = _native.LENS_EQUIDISTANT, 3.0, 4.0
    return d


@pytest.mark.parametrize("elem_bytes", [0, 3, 16])
def test_px_entry_points_refuse_other_element_widths(elem_bytes):
    lib = _native.load()
    d = _src_desc(_native.KIND_CAMERA)
    assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, elem_bytes, FAKE, 4, 4, FAKE, FAKE, None) == \
        _native.PB_ERR_UNSUPPORTED
    assert b"elem_bytes" in lib.pb_last_error()
    assert lib.pb_plan_remap_px(FAKE, elem_bytes, FAKE, 0, FAKE, 0, 1, None) == _native.PB_ERR_UNSUPPORTED
    assert b"elem_bytes" in lib.pb_last_error()
    assert lib.pb_plan_remap_rows_px(FAKE, elem_bytes, FAKE, FAKE, 0, 1, None) == _native.PB_ERR_UNSUPPORTED
    assert b"elem_bytes" in lib.pb_last_error()


def test_px_entry_points_refuse_null_pointers():
    lib = _native.load()
    d = _src_desc(_native.KIND_CAMERA)
    for e in (1, 2, 4, 8):
        assert lib.pb_plan_remap_px(None, e, FAKE, 0, FAKE, 0, 1, None) == _native.PB_ERR_INVALID_ARGUMENT
        assert b"null" in lib.pb_last_error()  # a null plan
        assert lib.pb_plan_remap_rows_px(None, e, FAKE, FAKE, 0, 1, None) == _native.PB_ERR_INVALID_ARGUMENT
        assert b"null" in lib.pb_last_error()
        assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, e, FAKE, 4, 4, None, FAKE, None) == \
            _native.PB_ERR_INVALID_ARGUMENT
        assert b"null" in lib.pb_last_error()
        assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, e, None, 4, 4, FAKE, FAKE, None) == \
            _native.PB_ERR_INVALID_ARGUMENT
        assert lib.pb_gather_from_map_px(None, 3, e, FAKE, 4, 4, FAKE, FAKE, None) == _native.PB_ERR_INVALID_ARGUMENT


def test_px_refuses_a_wide_double_fisheye_source():
    lib = _native.load()
    d = _src_desc(_native.KIND_DOUBLE)
    for e in (2, 4, 8):
        assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, e, FAKE, 4, 4, FAKE, FAKE, None) == \
            _native.PB_ERR_UNSUPPORTED
        assert b"double-fisheye" in lib.pb_last_error()


def test_px_refuses_misaligned_pointers():
    lib = _native.load()
    d = _src_desc(_native.KIND_CAMERA)
    odd = ctypes.c_void_p(257)
    for e in (2, 4, 8):
        assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, e, FAKE, 4, 4, odd, FAKE, None) == \
            _native.PB_ERR_INVALID_ARGUMENT
        assert b"multiple of elem_bytes" in lib.pb_last_error()
        assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, e, FAKE, 4, 4, FAKE, odd, None) == \
            _native.PB_ERR_INVALID_ARGUMENT
        assert b"multiple of elem_bytes" in lib.pb_last_error()
    d.kind = _native.KIND_EQUIRECT
    assert lib.pb_gather_from_map_px(ctypes.byref(d), 3, 4, FAKE, 4, 4, ctypes.c_void_p(258), FAKE, None) == \
        _native.PB_ERR_INVALID_ARGUMENT


def test_elem_bytes_table():
    import torch

    want = {np.bool_: 1, np.int8: 1, np.uint8: 1, np.int16: 2, np.uint16: 2, np.float16: 2, np.int32: 4,
            np.uint32: 4, np.float32: 4, np.int64: 8, np.uint64: 8, np.float64: 8}
    for dtype, width in want.items():
        assert engine.elem_bytes(np.zeros((2, 2, 3), dtype)) == width, dtype
    for dtype, width in ((torch.bool, 1), (torch.int8, 1), (torch.uint8, 1), (torch.int16, 2), (torch.float16, 2),
                         (torch.bfloat16, 2), (torch.int32, 4), (torch.float32, 4), (torch.int64, 8),
                         (torch.float64, 8), (torch.uint16, 2), (torch.uint32, 4), (torch.uint64, 8)):
        assert engine.elem_bytes(torch.zeros((2, 2), dtype=dtype)) == width, dtype
    assert set(engine.ELEM_BYTES) == {"bool", "int8", "uint8", "int16", "uint16", "float16", "bfloat16", "int32",
                                      "uint32", "float32", "int64", "uint64", "float64"}


@pytest.mark.parametrize("dtype", [np.complex128, object, np.dtype([("a", np.int32)]), np.dtype(">f4")])
def test_other_dtypes_are_refused_by_name(dtype):
    image = np.zeros((4, 4, 3), dtype=dtype)
    with pytest.raises(NotImplementedError, match=re.escape(str(image.dtype))):
        engine.elem_bytes(image)


def test_complex_torch_tensor_is_refused():
    import torch

    with pytest.raises(NotImplementedError, match="complex64"):
        engine.elem_bytes(torch.zeros((4, 4), dtype=torch.complex64))


@pytest.mark.parametrize("dtype", [np.float32, np.uint16, np.int8, np.bool_])
def test_wide_double_fisheye_source_is_refused_before_device_work(dtype, monkeypatch):
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage, PanoramaImage

    def no_device(*args, **kwargs):
        raise AssertionError("device work before the dtype check")

    monkeypatch.setattr(engine, "_torch", no_device)
    src = DoubleCameraImage(np.zeros((16, 32, 3), dtype), 3.4, pb_lens.equidistant())
    pano = PanoramaImage(np.zeros((16, 32, 3), np.uint8))
    with pytest.raises(NotImplementedError, match="double-fisheye source must be uint8"):
        src.process_coordinate_map(pano.get_coordinate_map())
    with pytest.raises(NotImplementedError, match="double-fisheye source must be uint8"):
        src.process_coordinate_map(np.zeros((4, 4, 3), np.float64))
