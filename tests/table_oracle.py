"""The NumPy oracle of a user-defined lens (a ``Lens`` of user callables, PB_LENS_TABLE): oracle/numpy_port.py
with every per-pixel lens evaluation replaced by the linear interpolation of the table the product built,
restated from ``lens_table_at`` (csrc/pb_device.cuh).  The library is built with -fmad=false, so NumPy
reproduces that interpolation bit for bit and the kernels can be held to the oracle's exact pixels.
``oracle/`` itself is unchanged: the lens functions of numpy_port are patched for the geometries whose
"lens" is a ``TableLens``, inside ``patched()``.

The focal distance comes from the callable, as ``CameraImage._compute_f_distance`` derives it (one scalar
call, as the reference makes it); every per-pixel ``lens_forward`` / ``lens_inverse`` goes through a
table -- or, for ``per_pixel="callable"``, through the user's function itself: the reference's own
result, which the table follows to its interpolation error."""

from __future__ import annotations

import contextlib
import warnings

import numpy as np

from oracle import numpy_port


def table_at(table, x_max, x):
    """lens_table_at of pb_device.cuh: scale = (n - 1) / x_max as upload_lens_tables computes it,
    t = x * scale clamped below at 0, i = trunc(t) (n - 2 where t >= n - 1), fr = min(t - i, 1),
    a + (b - a) * fr; NaN passes through."""
    table = np.asarray(table, dtype=np.float64)
    n = table.size
    scale = np.float64(n - 1) / np.float64(x_max)
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(all="ignore"):
        t = x * scale
        t = np.where(t < 0.0, 0.0, t)
        nan = np.isnan(x)
        top = t >= n - 1
        i = np.where(top, n - 2, np.trunc(np.where(nan | top, 0.0, t))).astype(np.int64)
        fr = np.minimum(t - i.astype(np.float64), 1.0)
        a, b = table[i], table[i + 1]
        out = a + (b - a) * fr
    return np.where(nan, x, out)


class TableLens:
    """A user-defined lens as the oracle sees it.

    forward / reverse: the user's callables.  source: (table, x_max) of the forward function (what a
    source of this lens evaluates per pixel), output: (table, x_max) of the reverse function (what an
    output evaluates); None where the lens is not used on that side.  per_pixel: "table" (what the
    kernels compute) or "callable" (the reference's evaluation)."""

    def __init__(self, forward, reverse, source=None, output=None, per_pixel="table"):
        if per_pixel not in ("table", "callable"):
            raise ValueError(per_pixel)
        self.forward, self.reverse = forward, reverse
        self.source, self.output = source, output
        self.per_pixel = per_pixel

    def with_per_pixel(self, per_pixel):
        return TableLens(self.forward, self.reverse, self.source, self.output, per_pixel)

    def forward_px(self, theta):
        if self.per_pixel == "callable":
            return _call(self.forward, theta)
        return table_at(self.source[0], self.source[1], theta)

    def reverse_px(self, d):
        if self.per_pixel == "callable":
            return _call(self.reverse, d)
        return table_at(self.output[0], self.output[1], d)

    def __repr__(self):
        sizes = [None if s is None else s[0].size for s in (self.source, self.output)]
        return f"TableLens(per_pixel={self.per_pixel}, samples={sizes})"


def _call(fn, x):
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return np.asarray(fn(np.asarray(x, dtype=np.float64)), dtype=np.float64)


_ORIGINAL = {name: getattr(numpy_port, name) for name in ("lens_forward", "lens_inverse", "focal_distance")}


def _lens_forward(lens, theta):
    if isinstance(lens, TableLens):
        return lens.forward_px(theta)
    return _ORIGINAL["lens_forward"](lens, theta)


def _lens_inverse(lens, d):
    if isinstance(lens, TableLens):
        return lens.reverse_px(d)
    return _ORIGINAL["lens_inverse"](lens, d)


def _focal_distance(geom):
    lens = geom.get("lens")
    if isinstance(lens, TableLens):  # magnitude / forward(fov / 2), the callable on a Python float
        magnitude = geom.get("magnitude") if geom["kind"] == "camera" else None
        if magnitude is None:
            magnitude = geom["height"] / 2.0
        return magnitude / lens.forward(geom["fov"] / 2)
    return _ORIGINAL["focal_distance"](geom)


@contextlib.contextmanager
def patched():
    """numpy_port (and with it helpers.stable_pixel_mask, typed_oracle.sample_double, coordinate_map)
    evaluates TableLens geometries through their tables; built-in lens names are untouched."""
    saved = {name: getattr(numpy_port, name) for name in _ORIGINAL}
    numpy_port.lens_forward, numpy_port.lens_inverse = _lens_forward, _lens_inverse
    numpy_port.focal_distance = _focal_distance
    try:
        yield
    finally:
        for name, fn in saved.items():
            setattr(numpy_port, name, fn)


def geom_of(image, per_pixel="table"):
    """The oracle's geometry dict of a product image (CameraImage, DoubleCameraImage, PanoramaImage),
    with the lens tables the product built for it on both sides (``_source_geometry`` /
    ``_output_geometry``) when its lens is user-defined."""
    from photonbend_b200 import _native
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, _frame_shape

    h, w = _frame_shape(image.image)
    if not isinstance(image, (CameraImage, DoubleCameraImage)):
        return {"kind": "equirect", "height": h, "width": w}
    src, out = image._source_geometry(), image._output_geometry()
    if src.lens == _native.LENS_TABLE:
        lens = TableLens(image.forward_lens, image.reverse_lens, (src.table, src.table_max),
                         (out.table, out.table_max), per_pixel)
    else:
        lens = _lens_name(src.lens)
    if isinstance(image, DoubleCameraImage):
        return {"kind": "double", "height": h, "width": w, "lens": lens, "fov": float(image.sensor_fov)}
    return {"kind": "camera", "height": h, "width": w, "lens": lens, "fov": float(image.fov),
            "magnitude": float(image.magnitude)}


def _lens_name(ident):
    from photonbend_b200 import _native

    for name in numpy_port.LENS_NAMES:
        if getattr(_native, "LENS_" + name.upper()) == ident:
            return name
    raise KeyError(ident)


def blended_mask(sg, cmap):
    """Double-fisheye source: the output pixels whose value blends a sample of each lens (both
    truncated positions inside their half, ray valid) -- numpy_port.sample_double's indices, so a
    table lens's own; the pixels the 1-LSB blend class may touch (helpers.Oracle)."""
    h, w = sg["height"], sg["width"]
    wl = w // 2
    invalid = cmap[:, :, 2] != 0.0
    lat_l = cmap[:, :, 0]
    lat_r = (lat_l * -1) + np.pi
    lon = cmap[:, :, 1]
    ok = ~invalid
    for lat, hw in ((lat_l, wl), (lat_r, w - wl)):
        f = numpy_port.focal_distance({"kind": "camera", "height": h, "width": hw, "lens": sg["lens"],
                                       "fov": sg["fov"], "magnitude": None})
        px, py = numpy_port._camera_pixel_positions(lat, lon, sg["lens"], f, h, hw)
        ok &= (px >= 0) & (px < hw) & (py >= 0) & (py < h)
    return ok


def source_coordinates(sg, cmap):
    """float64 (x, y) source coordinates of a camera source along ``cmap`` before truncation
    (numpy_port._camera_pixel_positions without the cast), and the radius in pixels."""
    h, w = sg["height"], sg["width"]
    f = numpy_port.focal_distance(sg)
    with np.errstate(all="ignore"):
        dist = numpy_port.lens_forward(sg["lens"], cmap[:, :, 0]) * f
        p = np.exp(cmap[:, :, 1] * 1j) * dist
        return p.real + (w / 2 - 0.5), (p.imag * (-1)) + (h / 2 - 0.5), dist
