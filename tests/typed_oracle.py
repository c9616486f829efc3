"""The NumPy oracle of a double-fisheye source blended in its own dtype
(DoubleCameraImage(..., keep_dtype=True)): oracle/numpy_port.py's sample_double, the reference's
projection.py:408-462, with its final cast to uint8 replaced by a cast to another type, and the
cast table that cast follows.  Shared by the tests and profiles/double_dtype_bench.py."""

from __future__ import annotations

import numpy as np

from oracle import numpy_port


def cast_x86(values, dtype: str):
    """float64 array -> ``dtype`` the way ``values.astype(dtype)`` does on x86-64, restated with
    explicit rules, so that it is defined where NumPy's own result is not (uint32 beyond +-2^32 casts
    differently depending on the array's length) and for bfloat16, which NumPy lacks (torch's cast:
    float64 -> float32 -> bfloat16, both to nearest even; returned as its uint16 bit patterns):

      uint8 / int8 / uint16 / int16   truncate to int32 (cvttsd2si), keep the low bits; NaN, |v| >= 2^31 -> 0
      int32                           truncate; NaN and out of range -> INT32_MIN
      int64                           truncate; NaN and |v| >= 2^63 -> INT64_MIN
      uint32                          truncate to int64 (as above), keep the low 32 bits
      uint64                          v < 2^63 or NaN: truncate to int64 (negatives wrap);
                                      else truncate v - 2^63 and xor 2^63
      float32 / float16               one rounding to nearest even (float16 straight from float64)
      bool                            v != 0
    """
    v = np.asarray(values, dtype=np.float64)
    two63 = 9223372036854775808.0

    def trunc64(x):  # int64 truncation, INT64_MIN where cvttsd2si overflows (NaN too)
        ok = (x >= -two63) & (x < two63)
        return np.where(ok, np.trunc(np.where(ok, x, 0.0)).astype(np.int64), np.int64(-2**63))

    if dtype in ("uint8", "int8", "uint16", "int16"):
        ok = np.abs(v) < 2147483648.0
        t = np.where(ok, np.trunc(np.where(ok, v, 0.0)), 0.0).astype(np.int64)
        return t.astype(dtype)  # (int64 -> narrower integer keeps the low bits)
    if dtype == "int32":
        ok = (v > -2147483649.0) & (v < 2147483648.0)
        return np.where(ok, np.trunc(np.where(ok, v, 0.0)), -2147483648.0).astype(np.int32)
    if dtype == "int64":
        return trunc64(v)
    if dtype == "uint32":
        return (trunc64(v) & 0xFFFFFFFF).astype(np.uint32)
    if dtype == "uint64":
        big = v >= two63
        small = trunc64(v).view(np.uint64)
        large = trunc64(np.where(big, v - two63, 0.0)).view(np.uint64) ^ np.uint64(1 << 63)
        return np.where(big, large, small)
    if dtype == "float32":
        return v.astype(np.float32)
    if dtype == "float16":
        return v.astype(np.float16)
    if dtype == "float64":
        return v.copy()
    if dtype == "bool":
        return v != 0.0
    if dtype == "bfloat16":
        with np.errstate(all="ignore"):
            bits = v.astype(np.float32).view(np.uint32).astype(np.uint64)
        rounded = (bits + 0x7FFF + ((bits >> 16) & 1)) >> 16
        nan = np.isnan(v)
        return np.where(nan, (bits >> 16) | 0x40, rounded).astype(np.uint16)
    raise KeyError(dtype)


def sample_double(geom: dict, image, cmap, dtype: str):
    """numpy_port.sample_double (reference projection.py:408-462) with the float64 blend cast by
    cast_x86(blend, dtype) instead of astype(uint8); ``image`` (H, W, C) of any dtype whose values
    float64 holds (bfloat16 images as the float32 values they hold)."""
    hs, ws = image.shape[:2]
    wl = ws // 2
    fov = geom["fov"]
    ref = (fov / 2) - (np.pi / 2)
    lo = np.pi / 2 - ref
    hi = np.pi / 2 + ref
    span = 2.0 * ref
    safety = numpy_port.deg2rad(0.5)

    invalid = cmap[:, :, 2] != 0.0
    lon = cmap[:, :, 1]
    lat_l = cmap[:, :, 0]
    lat_r = np.copy(lat_l)
    lat_r *= -1
    lat_r += np.pi

    img_l = image[:, :wl]
    img_r = np.copy(image[:, wl:])[:, ::-1]
    sub = {"kind": "camera", "lens": geom["lens"], "fov": fov, "magnitude": None}
    f_l = numpy_port.focal_distance(dict(sub, height=img_l.shape[0], width=img_l.shape[1]))
    f_r = numpy_port.focal_distance(dict(sub, height=img_r.shape[0], width=img_r.shape[1]))
    pix_l = numpy_port._sample_camera_arrays(img_l, geom["lens"], f_l, lat_l, lon, invalid)
    pix_r = numpy_port._sample_camera_arrays(img_r, geom["lens"], f_r, lat_r, lon, invalid)

    def weight(lat):
        with np.errstate(all="ignore"):
            band = np.logical_and(lat >= lo, lat <= (hi + safety))
            wgt = (lat - hi) / span * -1
        wgt[np.logical_not(band)] = 1.0
        return np.expand_dims(wgt, 2)

    with np.errstate(all="ignore"):
        blend = pix_l.astype(np.float64) * weight(lat_l) + pix_r.astype(np.float64) * weight(lat_r)
        out = cast_x86(blend, dtype)
    out[invalid] = 0
    return out
