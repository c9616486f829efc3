"""The C-ABI library loads on a CPU-only box and exports every symbol include/pb_remap.h
declares; argument errors come back as codes + messages without touching a GPU."""

import ctypes
import os
import re

from conftest import REPO


def _declared_functions():
    with open(os.path.join(REPO, "include", "pb_remap.h")) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pb_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    from photonbend_b200 import _native

    declared = _declared_functions()
    assert declared, "no functions found in include/pb_remap.h"
    assert sorted(_native.EXPORTS) == declared


def test_library_exports_every_declared_symbol():
    from photonbend_b200 import _native

    lib = _native.load()
    for name in _declared_functions():
        assert hasattr(lib, name), name
    assert lib.pb_version() == _native.PB_ABI_VERSION == 2


def test_struct_layout_matches_header():
    from photonbend_b200 import _native

    assert ctypes.sizeof(_native.ImageDesc) == 56  # 4 x int32, 2 x double, pointer, 2 x int32, double
    assert _native.ImageDesc.lens_table.offset == 32 and _native.ImageDesc.lens_table_max.offset == 48
    assert ctypes.sizeof(_native.RemapDesc) == 2 * 56 + 8 + _native.PB_MAX_ROTATIONS * 9 * 8
    assert _native.RemapDesc.rotations.offset == 120


def test_launch_families_match_header():
    """pb_debug_launch_counts: the PB_LAUNCH_* enum and _native.LAUNCH_FAMILIES name the same
    families in the same order, and the families add up to pb_kernel_launches()."""
    from photonbend_b200 import _native

    with open(os.path.join(REPO, "include", "pb_remap.h")) as fh:
        text = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    values = {name: int(v) for name, v in re.findall(r"\bPB_LAUNCH_([A-Z0-9_]+)\s*=\s*(\d+)", text)}
    n = values.pop("FAMILIES")
    assert sorted(values.values()) == list(range(n))
    assert tuple(name.lower() for name in sorted(values, key=values.get)) == _native.LAUNCH_FAMILIES
    lib = _native.load()
    assert lib.pb_debug_launch_counts(None, 0) == n
    short = (ctypes.c_int64 * 2)(-1, -1)
    assert lib.pb_debug_launch_counts(short, 1) == n and short[1] == -1  # writes no more than capacity
    counts = _native.launch_counts()
    assert min(counts.values()) >= 0 and sum(counts.values()) == lib.pb_kernel_launches()


def test_argument_errors_need_no_gpu():
    from photonbend_b200 import _native

    lib = _native.load()
    d = _native.RemapDesc()
    assert lib.pb_remap_u8(ctypes.byref(d), None, 0, None, 0, 1, None) == _native.PB_ERR_INVALID_ARGUMENT
    assert b"null" in lib.pb_last_error()
    fake = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    d.out.kind, d.out.height, d.out.width = _native.KIND_EQUIRECT, 0, 10
    assert lib.pb_remap_u8(ctypes.byref(d), fake, 0, fake, 0, 1, None) == _native.PB_ERR_INVALID_ARGUMENT
    assert b"positive" in lib.pb_last_error()
    d.out.height = 8
    d.src.kind, d.src.height, d.src.width, d.src.lens = _native.KIND_CAMERA, 8, 8, 99
    assert lib.pb_remap_u8(ctypes.byref(d), fake, 0, fake, 0, 1, None) == _native.PB_ERR_INVALID_ARGUMENT
    assert b"lens" in lib.pb_last_error()
    d.src.lens, d.channels, d.n_rotations = 0, 3, _native.PB_MAX_ROTATIONS + 1
    assert lib.pb_remap_u8(ctypes.byref(d), fake, 0, fake, 0, 1, None) == _native.PB_ERR_TOO_MANY_ROTATIONS
    d.n_rotations, d.channels = 0, 9
    assert lib.pb_remap_u8(ctypes.byref(d), fake, 0, fake, 0, 1, None) == _native.PB_ERR_UNSUPPORTED
    d.channels = 3
    assert lib.pb_remap_u8(ctypes.byref(d), fake, 0, fake, 0, 0, None) == _native.PB_OK  # zero frames: nothing to do
    img = _native.ImageDesc()
    img.kind, img.height, img.width = _native.KIND_DOUBLE, 10, 11
    assert lib.pb_output_width(ctypes.byref(img)) == 10
    handle = ctypes.c_void_p()
    assert lib.pb_plan_create(None, None, ctypes.byref(handle)) == _native.PB_ERR_INVALID_ARGUMENT
    lib.pb_plan_destroy(None)  # destroying nothing is allowed


# ------------------------------------------------------------------ libpbio.so (include/pb_io.h)


def _declared_io_functions():
    with open(os.path.join(REPO, "include", "pb_io.h")) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pb_io_[a-z0-9_]+)\s*\(", text)))


def test_io_header_binding_and_library_agree():
    from photonbend_b200.utils import image_io

    declared = _declared_io_functions()
    assert declared and sorted(image_io.EXPORTS) == declared
    lib = image_io.load_codec()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pb_io_version() == 1


def test_io_argument_errors_need_no_gpu():
    from photonbend_b200.utils import image_io

    lib = image_io.load_codec()
    w, h, n = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    assert lib.pb_io_jpeg_info(None, 0, ctypes.byref(w), ctypes.byref(h), ctypes.byref(n)) == image_io.PB_IO_ERR_INVALID_ARGUMENT
    assert b"null" in lib.pb_io_last_error()
    size = ctypes.c_size_t(0)
    fake = ctypes.c_void_p(256)  # never dereferenced: validation fails first
    assert lib.pb_io_jpeg_encode_rgb_u8(fake, 0, 10, 75, 2, None, None, ctypes.byref(size)) == image_io.PB_IO_ERR_INVALID_ARGUMENT
    assert lib.pb_io_jpeg_encode_rgb_u8(fake, 10, 10, 0, 2, None, None, ctypes.byref(size)) == image_io.PB_IO_ERR_INVALID_ARGUMENT
    assert b"quality" in lib.pb_io_last_error()
    assert lib.pb_io_jpeg_encode_rgb_u8(fake, 10, 10, 75, 9, None, None, ctypes.byref(size)) == image_io.PB_IO_ERR_INVALID_ARGUMENT
    assert lib.pb_io_jpeg_decode_rgb_u8(None, 0, None, 1, 1, None) == image_io.PB_IO_ERR_INVALID_ARGUMENT


def test_codec_selection(monkeypatch):
    import pytest
    from photonbend_b200.utils import image_io

    monkeypatch.delenv("PHOTONBEND_B200_CODEC", raising=False)
    assert image_io.selected_codec() == "pil"
    monkeypatch.setenv("PHOTONBEND_B200_CODEC", "NVJPEG")
    assert image_io.selected_codec() == "nvjpeg"
    monkeypatch.setenv("PHOTONBEND_B200_CODEC", "turbo")
    with pytest.raises(ValueError):
        image_io.selected_codec()
