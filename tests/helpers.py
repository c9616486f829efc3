"""Bridges between the plain geometry dicts (tests, oracle, workloads) and the product's API."""

from __future__ import annotations

import numpy as np


def product_image(geom: dict, array):
    """photonbend_b200 projection image for a geometry dict."""
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, PanoramaImage

    if geom["kind"] == "equirect":
        return PanoramaImage(array)
    lens = getattr(pb_lens, geom["lens"])()
    if geom["kind"] == "camera":
        return CameraImage(array, geom["fov"], lens, magnitude=geom.get("magnitude"))
    return DoubleCameraImage(array, geom["fov"], lens)


def product_map(out_geom: dict, rotations=()):
    """Lazy coordinate map of the product for (output geometry, rotations)."""
    from photonbend_b200.core.rotation import Rotation

    dst = product_image(out_geom, np.zeros((out_geom["height"], out_geom["width"], 3), np.uint8))
    cmap = dst.get_coordinate_map()
    for pyr in rotations:
        cmap = Rotation(*pyr).rotate_coordinate_map(cmap)
    return cmap


def product_remap(out_geom: dict, rotations, src_geom: dict, image):
    """The reference's three-call protocol through the product (one fused CUDA launch)."""
    return product_image(src_geom, image).process_coordinate_map(product_map(out_geom, rotations))


def remap_launches(fn):
    """Run fn() -> (its result, {kernel family: grids launched}) for the kernels the library launched
    during the call (pb_debug_launch_counts), without the plan-time kernels of a first call."""
    from photonbend_b200 import _native

    before = _native.launch_counts()
    result = fn()
    after = _native.launch_counts()
    return result, {k: after[k] - before[k] for k in after if k != "plan" and after[k] != before[k]}


def attribute_mismatches(got, want, image, idx):
    """Classify the pixels where ``got`` != ``want``.

    idx: int64 (H, W, 2) source offsets from oracle.c_port.source_index (-1 = none).
    Returns (n_bad, n_index_flip, n_lsb, n_unexplained):
      index flip  -- got equals the source pixel one step (x or y, either slot) away from the
                     oracle's index, i.e. the truncated coordinate fell on the other side of an
                     integer boundary;
      lsb         -- every channel within 1 of the oracle (float64 blend truncation).
    """
    got = np.asarray(got)
    want = np.asarray(want)
    diff = (got != want).reshape(got.shape[0], got.shape[1], -1).any(axis=2)
    ys, xs = np.nonzero(diff)
    hs, ws = image.shape[:2]
    flat = image.reshape(hs * ws, -1)
    n_flip = n_lsb = n_unexplained = 0
    for y, x in zip(ys, xs):
        g = got[y, x].astype(np.int16).reshape(-1)
        w = want[y, x].astype(np.int16).reshape(-1)
        if np.abs(g - w).max() <= 1:
            n_lsb += 1
            continue
        explained = False
        for slot in (0, 1):
            o = int(idx[y, x, slot])
            if o < 0:
                continue
            for step in (-1, 1, -ws, ws, -ws - 1, -ws + 1, ws - 1, ws + 1):
                n = o + step
                if 0 <= n < hs * ws and np.array_equal(flat[n].astype(np.int16), g):
                    explained = True
        if not explained and not g.any():
            # black instead of a pixel (or vice versa): the coordinate crossed the image border
            explained = True
        if explained:
            n_flip += 1
        else:
            n_unexplained += 1
    return len(ys), n_flip, n_lsb, n_unexplained


def stable_pixel_mask(src_geom: dict, image, cmap, ulps: float = 8.0):
    """Pixels whose reference value does not depend on the last few ulps of the ray angles.

    The reference truncates float64 coordinates to pixel indices, so a pixel whose coordinate
    sits within rounding noise of an integer boundary (or of the lat == pi row wrap of a
    panorama, or of a blend-band edge) gets a value that depends on the libm in use -- NumPy's
    SIMD kernels on the reference side, CUDA's on ours (both 1-2 ulp accurate, neither correctly
    rounded).  Degenerate geometries (a 360-degree stereographic lens has an infinite image
    radius) put whole regions into that state.  The mask is computed with the oracle itself: the
    final coordinate map is nudged by +-``ulps`` units in the last place in latitude and in
    longitude, and a pixel is stable when every nudged map gives the same pixel.
    """
    from oracle import numpy_port

    base = numpy_port.sample(src_geom, image, cmap.copy())
    stable = np.ones(base.shape[:2], dtype=bool)
    for d_lat, d_lon in ((ulps, 0), (-ulps, 0), (0, ulps), (0, -ulps), (ulps, ulps), (-ulps, -ulps)):
        nudged = cmap.copy()
        with np.errstate(all="ignore"):
            nudged[:, :, 0] += d_lat * np.spacing(np.abs(nudged[:, :, 0]))
            nudged[:, :, 1] += d_lon * np.spacing(np.abs(nudged[:, :, 1]))
        other = numpy_port.sample(src_geom, image, nudged)
        stable &= (other.reshape(base.shape[0], base.shape[1], -1) ==
                   base.reshape(base.shape[0], base.shape[1], -1)).all(axis=2)
    return stable
