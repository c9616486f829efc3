"""Bridges between the plain geometry dicts (tests, oracle, workloads) and the product's API."""

from __future__ import annotations

import warnings

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


class Oracle:
    """Output frames of one geometry against the NumPy oracle: bit-exact on the pixels whose
    reference value does not hang on the last ulps of libm.  On those, a double-fisheye source may
    differ by the 1-LSB blend class only: a float64 blend v0 w0 + v1 w1 whose exact value is an
    integer truncates to v or v - 1 on the last ulp of the weights.  Only pixels that blend two
    source pixels can do that.  On noise frames 3 / 256 of them are exposed and the class stays
    below 2e-4 of the pixels (checked over all the frames of a test, see lsb_share); on a flat frame
    every blended pixel is.  A user-defined lens is held to the same rule: its geometry dict carries
    a tests/table_oracle.TableLens, and the oracle (under table_oracle.patched()) interpolates the
    tables the product built, as the kernels do.

    Besides the pixels stable_pixel_mask finds, a camera or double-fisheye output has
    pixels whose lens latitude sits within a few ulps of fov / 2 (a default magnitude puts whole
    pixels exactly on it): whether the reference marks them invalid hangs on the last ulp of its
    lens inverse, which nudging the final map does not reach."""

    def __init__(self, og, rots, sg):
        from oracle import c_port

        self.sg = sg
        self.cmap = oracle_map(og, rots)
        self.fov_edge = None
        if og["kind"] != "equirect":
            lat = oracle_map(og, ())[:, :, 0]
            if og["kind"] == "double":
                lat[:, og["width"] // 2:] = np.pi - lat[:, og["width"] // 2:]  # the right lens's own latitude
            self.fov_edge = np.abs(lat - og["fov"] / 2) <= 8 * np.spacing(np.pi)
        self.blended = None
        if sg["kind"] == "double" and all(isinstance(g.get("lens", ""), str) for g in (og, sg)):
            self.blended = (c_port.source_index(og, rots, sg) >= 0).all(axis=2)
        elif sg["kind"] == "double":  # a user lens: the table oracle's own indices (c_port knows the names only)
            import table_oracle

            self.blended = table_oracle.blended_mask(sg, self.cmap)
        self.n_lsb = self.n_px = 0  # 1-LSB pixels and pixels of the frames that are not flat

    def check(self, got, frame, cid):
        """-> (differing pixels, pixels, degenerate)"""
        bad, px, degenerate, lsb = assert_like_oracle(got, frame, self.sg, self.cmap, cid, self.blended, self.fov_edge)
        if frame.min() != frame.max():
            self.n_lsb += lsb
            self.n_px += px
        return bad, px, degenerate

    def assert_lsb_share(self):
        assert self.n_lsb <= 2e-4 * self.n_px, (self.n_lsb, self.n_px)


def assert_like_oracle(got, frame, sg, cmap, cid, blended=None, fov_edge=None):
    """-> (differing pixels, pixels, degenerate, 1-LSB blend pixels); see _Oracle"""
    from oracle import numpy_port

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = numpy_port.sample(sg, frame, cmap.copy())
    assert got.shape == want.shape, cid
    n_px = want.shape[0] * want.shape[1]
    if np.array_equal(got, want):
        return 0, n_px, False, 0
    diff = (got != want).any(axis=2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        stable = stable_pixel_mask(sg, frame, cmap)
    if fov_edge is not None:
        stable &= ~fov_edge
    if (~stable).mean() > 0.01:
        assert not (diff & stable).any() or sg["kind"] == "double", cid
        return 0, 0, True, 0
    hard = diff & stable
    if hard.any():
        delta = np.abs(got.astype(np.int16) - want.astype(np.int16)).max(axis=2)
        assert sg["kind"] == "double" and delta[hard].max() == 1, (cid, int(hard.sum()), int(delta[hard].max()))
        assert blended[hard].all(), (cid, int((hard & ~blended).sum()))
    return int(diff.sum()), n_px, False, int(hard.sum())


def oracle_map(og, rots):
    from oracle import numpy_port

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return numpy_port.coordinate_map(og, rots)
