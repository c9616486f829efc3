"""ctypes front-end of oracle/pb_oracle.c (scalar float64 C restatement; row bands on a
thread pool -- ctypes releases the GIL).

TEST INFRASTRUCTURE ONLY -- the checker, never the product.  Geometry dicts are the same
as in oracle/numpy_port.py; the focal distance is derived there (with NumPy, exactly as the
reference derives it) and handed to C as a double.
"""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from . import numpy_port

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpboracle.so")

_KINDS = {"camera": 0, "double": 1, "equirect": 2}
_LENSES = {name: i for i, name in enumerate(numpy_port.LENS_NAMES)}
# numpy_port.LENS_NAMES order == the PBO_* lens enum in pb_oracle.c
assert numpy_port.LENS_NAMES == (
    "equidistant",
    "equisolid",
    "orthographic",
    "stereographic",
    "rectilinear",
    "thoby",
)


class _Image(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int32),
        ("lens", ctypes.c_int32),
        ("height", ctypes.c_int32),
        ("width", ctypes.c_int32),
        ("fov", ctypes.c_double),
        ("f_distance", ctypes.c_double),
    ]


def build(force: bool = False) -> str:
    """Compile libpboracle.so with the committed Makefile (gcc only)."""
    src = os.path.join(_HERE, "pb_oracle.c")
    stale = not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", "libpboracle.so"], check=True, capture_output=True)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.pbo_remap_u8.restype = ctypes.c_int
        _lib.pbo_coordinate_map_f64.restype = ctypes.c_int
        _lib.pbo_source_index_i64.restype = ctypes.c_int
    return _lib


def _describe(geom: dict) -> _Image:
    d = _Image()
    d.kind = _KINDS[geom["kind"]]
    d.height = int(geom["height"])
    d.width = int(geom["width"])
    if geom["kind"] == "equirect":
        d.lens, d.fov, d.f_distance = 0, 0.0, 0.0
    else:
        d.lens = _LENSES[geom["lens"]]
        d.fov = float(geom["fov"])
        d.f_distance = float(numpy_port.focal_distance(geom))
    return d


def _matrices(rotations):
    mats = [numpy_port.rotation_matrix(*pyr) for pyr in rotations]
    arr = np.ascontiguousarray(np.array(mats, dtype=np.float64).reshape(-1, 9))
    return len(mats), arr


def out_shape(geom: dict):
    w = geom["width"]
    if geom["kind"] == "double":
        w = 2 * (w // 2)
    return geom["height"], w


def _run_banded(call, r0, r1, threads):
    """Run ``call(a, b)`` over disjoint row bands of [r0, r1) on a thread pool."""
    threads = threads or len(os.sched_getaffinity(0))
    n_rows = r1 - r0
    if threads <= 1 or n_rows < 2 * threads:
        rc = call(r0, r1)
        if rc != 0:
            raise RuntimeError(f"oracle call failed ({rc})")
        return
    from concurrent.futures import ThreadPoolExecutor

    n_bands = min(n_rows, threads * 8)
    edges = [r0 + (n_rows * k) // n_bands for k in range(n_bands + 1)]
    with ThreadPoolExecutor(max_workers=threads) as pool:
        for rc in pool.map(lambda k: call(edges[k], edges[k + 1]), range(n_bands)):
            if rc != 0:
                raise RuntimeError(f"oracle call failed ({rc})")


def remap(out_geom, rotations, src_geom, image, rows=None, threads=0):
    """uint8 remap of ``image``; ``rows=(r0, r1)`` returns only that band of output rows.
    ``threads``: 0 = all cores this process may use, 1 = the scalar single-thread port."""
    image = np.ascontiguousarray(image, dtype=np.uint8)
    squeeze = image.ndim == 2
    channels = 1 if squeeze else image.shape[2]
    h, w = out_shape(out_geom)
    r0, r1 = (0, h) if rows is None else rows
    dst = np.empty((h, w, channels), dtype=np.uint8) if rows is None else None
    band = dst if dst is not None else np.empty((r1 - r0, w, channels), dtype=np.uint8)
    # C writes row i at offset i*w*channels: shift the base pointer for a band buffer
    base = band.ctypes.data - r0 * w * channels
    n, mats = _matrices(rotations)
    o, s = _describe(out_geom), _describe(dict(src_geom, height=image.shape[0], width=image.shape[1]))
    fn = lib().pbo_remap_u8

    def call(a, b):
        return fn(
            ctypes.byref(o),
            ctypes.c_int(n),
            mats.ctypes.data_as(ctypes.c_void_p),
            ctypes.byref(s),
            image.ctypes.data_as(ctypes.c_void_p),
            ctypes.c_int(channels),
            ctypes.c_void_p(base),
            ctypes.c_int(a),
            ctypes.c_int(b),
        )

    _run_banded(call, r0, r1, threads)
    return band[:, :, 0] if squeeze else band


def coordinate_map(out_geom, rotations=(), threads=0):
    h, w = out_shape(out_geom)
    cmap = np.empty((h, w, 3), dtype=np.float64)
    n, mats = _matrices(rotations)
    o = _describe(out_geom)
    fn = lib().pbo_coordinate_map_f64

    def call(a, b):
        return fn(
            ctypes.byref(o),
            ctypes.c_int(n),
            mats.ctypes.data_as(ctypes.c_void_p),
            cmap.ctypes.data_as(ctypes.c_void_p),
            ctypes.c_int(a),
            ctypes.c_int(b),
        )

    _run_banded(call, 0, h, threads)
    return cmap


def source_index(out_geom, rotations, src_geom, threads=0, rows=None):
    """int64 (H, W, 2): linear source pixel offsets (left/only, right) or -1 for black.
    ``rows=(r0, r1)`` returns only that band of output rows, (r1 - r0, W, 2)."""
    h, w = out_shape(out_geom)
    r0, r1 = (0, h) if rows is None else rows
    band = np.empty((r1 - r0, w, 2), dtype=np.int64)
    base = band.ctypes.data - r0 * w * 2 * 8  # C writes row i at offset i*w*2 int64s
    n, mats = _matrices(rotations)
    o, s = _describe(out_geom), _describe(src_geom)
    fn = lib().pbo_source_index_i64

    def call(a, b):
        return fn(
            ctypes.byref(o),
            ctypes.c_int(n),
            mats.ctypes.data_as(ctypes.c_void_p),
            ctypes.byref(s),
            ctypes.c_void_p(base),
            ctypes.c_int(a),
            ctypes.c_int(b),
        )

    _run_banded(call, r0, r1, threads)
    return band
