"""A double-fisheye source blended in its own dtype (DoubleCameraImage(..., keep_dtype=True)), the
parts that need no GPU: the cast table of tests/typed_oracle.py (cast_x86) against NumPy's and
torch's casts, its blend against oracle/numpy_port.py, the argument errors of the _typed entry
points, and the refusals of the Python layer."""

import ctypes
import warnings

import numpy as np
import pytest

import typed_oracle
from oracle import numpy_port
from photonbend_b200 import _native as N
from photonbend_b200 import engine

TWO63 = 2.0**63
EDGES = [np.nan, np.inf, -np.inf, 0.0, -0.0, 0.5, -0.5, 1.5, -1.5, 199.99999999999997, 255.5, 256.0, -1.0,
         2.0**31 - 0.5, 2.0**31 + 0.5, -(2.0**31) - 0.5, -(2.0**31) + 0.5, -(2.0**31), 2.0**31,
         2.0**40 + 3.5, -(2.0**40) - 3.5, 2.0**32 + 5.0, TWO63, -TWO63, TWO63 - 1024.0, 2.0**64, 2.0**53 + 2.0,
         1e300, -1e300, -70000.5, 70000.5, 65504.0, 65519.99, 65520.0,
         # float16 ties and the single-rounding cases: 2**-25 -> 0, 2**-25 + 2**-60 -> the smallest denormal
         2.0**-25, 2.0**-25 + 2.0**-60, 3 * 2.0**-25, 1.0 + 2.0**-11, 1.0 + 3 * 2.0**-11, 1.0 + 2.0**-11 + 2.0**-40,
         # float32 / bfloat16 ties and double roundings
         1.0 + 2.0**-24, 1.0 + 2.0**-8 + 2.0**-32, 1.0 + 2.0**-8, 1.0 + 3 * 2.0**-8, 3.4e38, 3.5e38, 1e-45, 1e-310]

INT_TYPES = ("uint8", "int8", "uint16", "int16", "int32", "uint32", "int64", "uint64")


def _astype(values, dtype):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return np.asarray(values, np.float64).astype(dtype)


@pytest.mark.parametrize("dtype", INT_TYPES + ("float16", "float32", "float64", "bool"))
def test_cast_table_matches_numpy(dtype):
    """cast_x86 restates NumPy's float64 casts on x86-64 rule by rule; uint32 against one-element
    casts, the only ones NumPy defines the same way for every value."""
    v = np.array(EDGES)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = typed_oracle.cast_x86(v, dtype)
        if dtype == "uint32":
            want = np.array([_astype([x], np.uint32)[0] for x in EDGES], np.uint32)
        else:
            want = _astype(v, dtype)
    assert got.dtype == want.dtype
    same = got == want
    if dtype.startswith("float"):
        same |= np.isnan(got) & np.isnan(want)
        same &= np.signbit(got) == np.signbit(want)
    assert same.all(), [(EDGES[i], got[i], want[i]) for i in np.nonzero(~same)[0]]


def test_cast_table_bfloat16_matches_torch():
    """bfloat16: torch's CPU cast rounds twice (float64 -> float32 -> bfloat16); NaN payloads aside."""
    import torch

    v = np.array(EDGES)
    got = typed_oracle.cast_x86(v, "bfloat16")
    want = torch.tensor(v, dtype=torch.float64).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    nan = np.isnan(v)
    assert np.array_equal(got[~nan], want[~nan])
    assert ((got[nan] & 0x7F80) == 0x7F80).all() and (got[nan] & 0x7F).all()
    # the double rounding is what tells the two apart
    assert got[EDGES.index(1.0 + 2.0**-8 + 2.0**-32)] == 0x3F80


@pytest.mark.parametrize("rotations", [(), ((0.3, -0.7, 1.1),)])
@pytest.mark.parametrize("fov_deg", [195, 180, 170, 180.00000000001])
def test_typed_oracle_with_the_uint8_cast_is_the_oracle(rotations, fov_deg):
    """typed_oracle.sample_double is numpy_port.sample_double with its cast replaced: cast to uint8
    it gives the oracle's bytes (blend band, zero-width band, negative range, huge weights), and a
    wider integer cast keeps the same low byte; a float cast keeps the image's dtype."""
    import typed_oracle as t

    sg = {"kind": "double", "height": 40, "width": 80, "lens": "equidistant", "fov": np.pi * fov_deg / 180}
    cmap = numpy_port.coordinate_map({"kind": "equirect", "height": 48, "width": 96}, rotations)
    img = np.random.default_rng(3).integers(0, 256, (40, 80, 3), dtype=np.uint8)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        u8 = numpy_port.sample_double(sg, img, cmap.copy())
        assert np.array_equal(t.sample_double(sg, img, cmap.copy(), "uint8"), u8)
        assert np.array_equal(t.sample_double(sg, img, cmap.copy(), "uint16").astype(np.uint8), u8)
        f = t.sample_double(sg, img, cmap.copy(), "float32")
    assert f.dtype == np.float32 and f.shape == u8.shape


# --------------------------------------------------------------------------- ABI argument errors

FAKE, ODD = 256, 257
_plans = {k: (ctypes.c_int32 * (1 << 14))(*([k] * (1 << 14))) for k in (-1, 1)}
OTHER_DEVICE = ctypes.addressof(_plans[-1])  # camera-like source on no device (see test_abi_argument_errors)
DOUBLE_SRC = ctypes.addressof(_plans[1])  # double-fisheye source, 1 output row, device 1
INVALID, UNSUPPORTED = N.PB_ERR_INVALID_ARGUMENT, N.PB_ERR_UNSUPPORTED
ALIGN_MSG = "pointer or stride not a multiple of elem_bytes"


def _image(kind=N.KIND_DOUBLE):
    d = N.ImageDesc()
    d.kind, d.height, d.width, d.lens, d.fov, d.f_distance = kind, 8, 16, N.LENS_EQUIDISTANT, 3.0, 4.0
    return d


F32 = N.ELEM_TYPES["float32"]
ROT = (ctypes.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
CASES = {
    "typed-unknown+null": (("pb_plan_remap_typed", (None, 13, FAKE, 0, FAKE, 0, 1, None)), UNSUPPORTED,
                           "pb_plan_remap_typed: unknown element type 13"),
    "typed-negative": (("pb_plan_remap_typed", (DOUBLE_SRC, -1, FAKE, 0, FAKE, 0, 1, None)), UNSUPPORTED,
                       "pb_plan_remap_typed: unknown element type -1"),
    "typed-null": (("pb_plan_remap_typed", (DOUBLE_SRC, F32, None, 0, FAKE, 0, 1, None)), INVALID,
                   "pb_plan_remap_typed: null pointer"),
    "typed-align": (("pb_plan_remap_typed", (DOUBLE_SRC, F32, ODD, 0, FAKE, 0, 1, None)), INVALID,
                    "pb_plan_remap_typed: " + ALIGN_MSG),
    "typed-align-stride": (("pb_plan_remap_typed", (DOUBLE_SRC, N.ELEM_TYPES["float64"], FAKE, 4, FAKE, 0, 1, None)),
                           INVALID, "pb_plan_remap_typed: " + ALIGN_MSG),
    "typed-double-zero-frames": (("pb_plan_remap_typed", (DOUBLE_SRC, F32, FAKE, 0, FAKE, 0, 0, None)), N.PB_OK, None),
    "typed-bool-odd": (("pb_plan_remap_typed", (DOUBLE_SRC, N.ELEM_TYPES["bool"], ODD, 3, ODD, 0, 0, None)), N.PB_OK,
                       None),
    "typed-device": (("pb_plan_remap_typed", (OTHER_DEVICE, F32, FAKE, 0, FAKE, 0, 1, None)), INVALID,
                     "pb_plan_remap_typed: plan belongs to another device"),
    "rows-unknown": (("pb_plan_remap_rows_typed", (None, 99, FAKE, FAKE, 0, 1, None)), UNSUPPORTED,
                     "pb_plan_remap_rows_typed: unknown element type 99"),
    "rows-null": (("pb_plan_remap_rows_typed", (DOUBLE_SRC, F32, FAKE, None, 0, 1, None)), INVALID,
                  "pb_plan_remap_rows_typed: null pointer"),
    "rows-align": (("pb_plan_remap_rows_typed", (DOUBLE_SRC, N.ELEM_TYPES["uint16"], FAKE, ODD, 0, 1, None)), INVALID,
                   "pb_plan_remap_rows_typed: " + ALIGN_MSG),
    "rows-outside": (("pb_plan_remap_rows_typed", (DOUBLE_SRC, F32, FAKE, FAKE, 0, 2, None)), INVALID,
                     "pb_plan_remap_rows_typed: rows outside the output image"),
    "rows-empty": (("pb_plan_remap_rows_typed", (DOUBLE_SRC, F32, FAKE, FAKE, 1, 1, None)), N.PB_OK, None),
    "frames-unknown": (("pb_plan_remap_frames_typed", (DOUBLE_SRC, 100, ROT, FAKE, 0, FAKE, 0, 1, None)), UNSUPPORTED,
                       "pb_plan_remap_frames_typed: unknown element type 100"),
    "frames-null-rotations": (("pb_plan_remap_frames_typed", (DOUBLE_SRC, F32, None, FAKE, 0, FAKE, 0, 1, None)),
                              INVALID, "pb_plan_remap_frames_typed: null pointer"),
    "frames-align": (("pb_plan_remap_frames_typed", (DOUBLE_SRC, F32, ROT, FAKE, 2, FAKE, 0, 1, None)), INVALID,
                     "pb_plan_remap_frames_typed: " + ALIGN_MSG),
    "frames-neg": (("pb_plan_remap_frames_typed", (DOUBLE_SRC, F32, ROT, FAKE, 0, FAKE, 0, -1, None)), INVALID,
                   "pb_plan_remap_frames_typed: negative n_frames"),
    "gather-unknown": (("pb_gather_from_map_typed", (None, 3, 77, FAKE, 4, 4, FAKE, FAKE, None)), UNSUPPORTED,
                       "pb_gather_from_map_typed: unknown element type 77"),
    "gather-null": (("pb_gather_from_map_typed", (ctypes.byref(_image()), 3, F32, None, 4, 4, FAKE, FAKE, None)),
                    INVALID, "pb_gather_from_map_typed: null pointer"),
    "gather-align": (("pb_gather_from_map_typed", (ctypes.byref(_image()), 3, F32, FAKE, 4, 4, FAKE, ODD, None)),
                     INVALID, "pb_gather_from_map_typed: " + ALIGN_MSG),
    "gather-empty": (("pb_gather_from_map_typed", (ctypes.byref(_image()), 3, F32, FAKE, 0, 4, FAKE, FAKE, None)),
                     N.PB_OK, None),
}


@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_typed_argument_error(case):
    (fn, args), code, want = CASES[case]
    lib = N.load()
    assert getattr(lib, fn)(*args) == code
    if want is not None:
        assert lib.pb_last_error().decode() == want


def test_px_still_refuses_a_wide_double_source_that_typed_takes():
    lib = N.load()
    assert lib.pb_plan_remap_px(DOUBLE_SRC, 4, FAKE, 0, FAKE, 0, 0, None) == UNSUPPORTED
    assert lib.pb_plan_remap_typed(DOUBLE_SRC, F32, FAKE, 0, FAKE, 0, 0, None) == N.PB_OK


def test_elem_type_codes_cover_every_accepted_dtype():
    assert set(N.ELEM_TYPES) == set(engine.ELEM_BYTES)
    assert sorted(N.ELEM_TYPES.values()) == list(range(len(N.ELEM_TYPES)))


# --------------------------------------------------------------------------- Python layer


def _no_device(monkeypatch):
    def no_device(*args, **kwargs):
        raise AssertionError("device work before the dtype check")

    monkeypatch.setattr(engine, "_torch", no_device)


@pytest.mark.parametrize("dtype", [np.float32, np.uint16, np.int8, np.bool_])
def test_default_still_refuses_before_device_work(dtype, monkeypatch):
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage, PanoramaImage

    _no_device(monkeypatch)
    src = DoubleCameraImage(np.zeros((16, 32, 3), dtype), 3.4, pb_lens.equidistant(), keep_dtype=False)
    pano = PanoramaImage(np.zeros((16, 32, 3), np.uint8))
    with pytest.raises(NotImplementedError, match="keep_dtype=True"):
        src.process_coordinate_map(pano.get_coordinate_map())


@pytest.mark.parametrize("dtype", [np.complex64, np.float128 if hasattr(np, "float128") else np.complex128])
def test_keep_dtype_refuses_unsupported_dtypes_by_name(dtype, monkeypatch):
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage, PanoramaImage

    _no_device(monkeypatch)
    src = DoubleCameraImage(np.zeros((16, 32, 3), dtype), 3.4, pb_lens.equidistant(), keep_dtype=True)
    pano = PanoramaImage(np.zeros((16, 32, 3), np.uint8))
    with pytest.raises(NotImplementedError, match=np.dtype(dtype).name):
        src.process_coordinate_map(pano.get_coordinate_map())


def test_keep_dtype_changes_no_descriptor_byte():
    """One cached plan serves both settings: the flag is a property of the calls."""
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage, PanoramaImage

    img = np.zeros((16, 32, 3), np.float32)
    keep = DoubleCameraImage(img, 3.4, pb_lens.equidistant(), keep_dtype=True)
    default = DoubleCameraImage(img, 3.4, pb_lens.equidistant())
    assert keep.keep_dtype and not default.keep_dtype
    rays = PanoramaImage(np.zeros((8, 16, 3), np.uint8)).get_coordinate_map().rays
    a = engine._build_remap_desc(rays, keep._source_geometry(), 3)
    b = engine._build_remap_desc(rays, default._source_geometry(), 3)
    assert bytes(a) == bytes(b)
    assert engine.typed_blend(keep._source_geometry(), img) == N.ELEM_TYPES["float32"]
    assert engine.typed_blend(keep._source_geometry(), img.astype(np.uint8)) is None
    assert engine.typed_blend(default._source_geometry(), img) is None
