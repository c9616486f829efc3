"""Edge values through the float-to-integer steps of the device remap.  GPU only.

The kernels restate NumPy's casts by hand: ``.astype(int)`` then the bounds test (trunc_index),
Python's ``%`` of a truncation (wrap_index, floor_mod, trunc_i64) and ``.astype(np.uint8)`` of the
double-fisheye blend and of map_projection (cast_u8: a 32-bit truncation on x86-64, 0 for NaN and
|v| >= 2^31).  The product's own geometry only feeds them latitudes in [0, pi] and longitudes in
[-pi, pi].  An explicit coordinate map is a public input, though, and the reference is defined on
any float64 map, so the tests here draw maps from menus of edge values (pixel boundaries and their
ulp neighbours, negative and huge coordinates, +-2^31 and 2^63 pixel units, infinities, NaNs with
payloads, signed-zero and NaN flags) and compare the device with oracle/numpy_port.py run on the
same array.

Where no libm is involved the result must be bit-exact: equirect sources (division, truncation,
modulo), map_projection, and camera / double sources through an equidistant lens at longitude
+-0.0 (cos 0 = 1, sin 0 = 0 in every library).  Elsewhere CUDA's sin / cos / atan2 may differ
from NumPy's in the last ulp, so pixels are compared where the reference's own value does not
hang on those ulps (helpers.stable_pixel_mask), and the share of such unstable pixels is bounded
per test so that it cannot hide a regression.
"""

import numpy as np
import pytest

import case_matrix
import helpers
from conftest import mismatch_report
from oracle import numpy_port

pytestmark = pytest.mark.gpu

rad = case_matrix.rad
ROT = ((0.3, -0.7, 1.1),)
# sensor fovs of a double source within 2e-13 rad of pi: the blend band 2 * (fov/2 - pi/2) nearly
# vanishes and the blend of the two lenses grows past the 32 bits of NumPy's uint8 cast
NEAR_180 = {
    "180.00000000001": rad(180.00000000001),
    "179.99999999999": rad(179.99999999999),
    "nextafter_up": float(np.nextafter(np.pi, np.inf)),
    "nextafter_down": float(np.nextafter(np.pi, 0.0)),
}
TINY = float(np.finfo(np.float64).smallest_subnormal)
NANS = np.array([0x7FF8000000000000, 0xFFF8000000000000, 0x7FF800000000BEEF, 0xFFF0000000000001, 0x7FF4000000000000],
                dtype=np.uint64).view(np.float64)
SPECIALS = np.concatenate([[0.0, -0.0, TINY, -TINY, 1e-310, -1e-310, np.inf, -np.inf, 1e300, -1e300], NANS])


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


# ------------------------------------------------------------------------------------ helpers


def _around(values, ulps=2):
    """values and their neighbours up to ``ulps`` units in the last place on both sides"""
    out = [np.asarray(values, dtype=np.float64)]
    up = down = out[0]
    for _ in range(ulps):
        up, down = np.nextafter(up, np.inf), np.nextafter(down, -np.inf)
        out += [up, down]
    return np.concatenate([o.ravel() for o in out])


def _huge(unit):
    """+-(2^31 + {0, 1, 7}), +-2^32 and +-2^63 coordinate units, and their ulp neighbours"""
    n = np.array([2.0**31, 2.0**31 + 1, 2.0**31 + 7, 2.0**31 - 1, 2.0**32, 2.0**63])
    return _around(np.concatenate([n, -n]) * unit, 1)


def _pick(rng, menus, shape, weights=None):
    """Each entry: one of ``menus`` at random (by ``weights``), then one value of it.  Values are
    copied bit for bit (NaN payloads and signs survive)."""
    menus = [np.asarray(m, dtype=np.float64).ravel() for m in menus]
    which = rng.choice(len(menus), size=shape, p=weights)
    out = np.empty(shape)
    for k, m in enumerate(menus):
        sel = which == k
        out[sel] = m[rng.integers(0, m.size, int(sel.sum()))]
    return out


def _flags(rng, shape):
    """mostly 0; -0.0 (valid) and 1, -1, a denormal, inf, NaN (all invalid)"""
    menu = [[0.0], [-0.0], [1.0], [-1.0], [TINY], [np.inf], NANS]
    return _pick(rng, menu, shape, [0.7, 0.1, 0.04, 0.04, 0.04, 0.04, 0.04])


def _stack(lat, lon, flag):
    return np.ascontiguousarray(np.stack([lat, lon, flag], axis=2))


def equirect_edge_map(seed, src_h, src_w, shape=(256, 320)):
    """Entries that land on, just beside and far beyond the row / column boundaries of an equirect
    source of src_h x src_w (latitude k * pi/src_h, longitude (k - src_w/2) * pi/(src_w/2))."""
    rng = np.random.default_rng(seed)
    seg_h, seg_w = np.pi / src_h, np.pi / (src_w / 2)
    rows = np.arange(-3, src_h + 4) * seg_h
    cols = (np.arange(-3, src_w + 4) - src_w / 2) * seg_w
    turns = np.array([1, -1, 3, -7, 1000, -123456, 10**9]) * 2 * np.pi
    lat = _pick(rng, [
        _around(rows), -seg_h * rng.uniform(0, 1, 64), [np.pi, np.nextafter(np.pi, 4), np.nextafter(np.pi, 0)],
        rng.uniform(-50, 0, 64), rng.uniform(np.pi, 50, 64), _huge(seg_h), SPECIALS], shape)
    lon = _pick(rng, [
        _around(cols), (cols[:, None] + turns[None, :]).ravel(), rng.uniform(-1e6, 1e6, 64),
        rng.uniform(-np.pi, np.pi, 64), _huge(seg_w), SPECIALS], shape)
    return _stack(lat, lon, _flags(rng, shape))


def camera_edge_map(seed, sg, shape=(192, 256)):
    """Entries for a camera source: pixel boundaries of an equidistant lens at longitude 0
    (x = lat * f + cx on k and k +- ulp, and in (-1, 0)), the rectilinear domain (below 0, at
    to_radians(89) and just past it), fov / 2, pi, far beyond, and the specials.  The first third
    of the rows has longitude +-0.0."""
    rng = np.random.default_rng(seed)
    f = numpy_port.focal_distance(sg)
    cx = sg["width"] / 2 - 0.5
    ks = np.arange(-2, sg["width"] + 3)
    lat = _pick(rng, [
        _around((ks - cx) / f), (-rng.uniform(0, 1, 64) - cx) / f, rng.uniform(0, sg["fov"] / 2 + 0.3, 64),
        rng.uniform(-0.5, 0, 64), _around([rad(89), sg["fov"] / 2, np.pi, 0.0]), rng.uniform(4, 1e4, 64),
        _huge(1 / f), SPECIALS], shape)
    lon = _pick(rng, [
        rng.uniform(-np.pi, np.pi, 64), _around([np.pi, -np.pi, np.pi / 2, -np.pi / 2]),
        rng.uniform(-1e5, 1e5, 64), [1e300, -1e300, 2.0**63], SPECIALS], shape)
    zero_rows = shape[0] // 3
    lon[:zero_rows] = np.where(rng.integers(0, 2, (zero_rows, shape[1])) == 1, 0.0, -0.0)
    return _stack(lat, lon, _flags(rng, shape))


def double_blend_edges(fov):
    """The blend band of a double source of sensor fov the way the reference derives it
    (projection.py:414-418): [lo, hi + safety] for the left lens, pi - that for the right one."""
    ref = (fov / 2) - (np.pi / 2)
    lo, hi = np.pi / 2 - ref, np.pi / 2 + ref
    top = hi + rad(0.5)
    return np.array([lo, hi, top, np.pi - lo, np.pi - hi, np.pi - top, np.pi / 2]), abs(ref)


def double_edge_map(seed, sg, shape=(192, 256)):
    """Entries for a double source: the blend band's edges and their ulp neighbours, latitudes
    inside a band of any width, pixel boundaries of the left lens at longitude 0, and the
    specials.  The first third of the rows has longitude +-0.0."""
    rng = np.random.default_rng(seed)
    half = dict(sg, kind="camera", width=sg["width"] // 2, magnitude=None)
    f = numpy_port.focal_distance(half)
    cx = half["width"] / 2 - 0.5
    edges, ref = double_blend_edges(sg["fov"])
    ks = np.arange(-2, half["width"] + 3)
    lat = _pick(rng, [
        _around(edges, 3), np.pi / 2 + rng.uniform(-3, 3, 256) * max(ref, 1e-15),
        rng.uniform(edges[0] - 0.01, edges[2] + 0.01, 64), rng.uniform(0, np.pi, 64), _around((ks - cx) / f),
        rng.uniform(-1, 0, 16), _huge(1 / f), SPECIALS], shape)
    lon = _pick(rng, [rng.uniform(-np.pi, np.pi, 64), rng.uniform(-1e5, 1e5, 64), SPECIALS], shape)
    zero_rows = shape[0] // 3
    lon[:zero_rows] = np.where(rng.integers(0, 2, (zero_rows, shape[1])) == 1, 0.0, -0.0)
    return _stack(lat, lon, _flags(rng, shape))


def stable_mask(src_geom, image, cmap):
    """helpers.stable_pixel_mask, with every entry whose latitude or longitude is not finite
    counted as stable: such an entry goes through no libm-dependent rounding (NaN and inf
    propagate the same way in every library), and the nudged maps of the helper turn inf into NaN,
    which would call exactly the class under test unstable."""
    image = np.asarray(image)
    stable = helpers.stable_pixel_mask(src_geom, image, cmap)
    return stable | ~np.isfinite(cmap[:, :, 0]) | ~np.isfinite(cmap[:, :, 1])


def compare(tag, got, want, exact, max_unstable):
    """got == want byte for byte wherever ``exact``; -> (pixels that must match, pixels allowed
    to differ, pixels that do differ among those).  The allowed share is bounded by ``max_unstable``."""
    want = np.asarray(want)
    gb = np.ascontiguousarray(np.asarray(got)).view(np.uint8).reshape(want.shape[0], want.shape[1], -1)
    wb = np.ascontiguousarray(want).view(np.uint8).reshape(gb.shape)
    diff = (gb != wb).any(axis=2)
    bad = diff & exact
    if bad.any():
        ys, xs = np.nonzero(bad)
        raise AssertionError(f"{tag}: {int(bad.sum())} pixels differ where they must not, e.g. "
                             f"{[(int(y), int(x)) for y, x in zip(ys[:5], xs[:5])]}")
    allowed = ~exact
    assert allowed.mean() <= max_unstable, (tag, float(allowed.mean()))
    return int(exact.sum()), int(allowed.sum()), int((diff & allowed).sum())


def _tally(counts, kind, c):
    t = counts.setdefault(kind, [0, 0, 0])
    for k in range(3):
        t[k] += c[k]


def _report(name, counts):
    for kind, (n_exact, n_allowed, n_diff) in counts.items():
        print(f"{name} {kind}: {n_exact} pixels bit-exact, {n_allowed} unstable pixels allowed to differ, "
              f"{n_diff} of them differ")


# ------------------------------------------------------------------------- near-180 sources


def _near_180_source(fov, width=672, channels=3):
    sg = {"kind": "double", "height": 336, "width": width, "lens": "equidistant", "fov": fov}
    h = sg["height"]
    flat = np.full((h, width, channels), 200, np.uint8)
    noise = case_matrix.case_image(sg, 9, channels)
    return sg, {"kind": "equirect", "height": 352, "width": 704}, [flat, noise]


@pytest.mark.parametrize("fov_name", list(NEAR_180))
def test_near_180_double_sources_rotated(torch_cuda, fov_name):
    """Rotated output through a near-180 double source: one frame (direct kernel) and a batch
    (tiled kernel with per-pixel rays), against the NumPy oracle on stable pixels."""
    torch = torch_cuda
    sg, og, frames = _near_180_source(NEAR_180[fov_name])
    cmap = numpy_port.coordinate_map(og, ROT)
    batch = helpers.product_image(sg, torch.from_numpy(np.stack(frames)).cuda()).process_coordinate_map(
        helpers.product_map(og, ROT)).cpu().numpy()
    counts = {}
    for k, frame in enumerate(frames):
        want = numpy_port.remap(og, ROT, sg, frame)
        stable = helpers.stable_pixel_mask(sg, frame, cmap)
        got = helpers.product_remap(og, ROT, sg, frame)
        _tally(counts, "single frame", compare((fov_name, "single", k), got, want, stable, 0.02))
        _tally(counts, "batch", compare((fov_name, "batch", k), batch[k], want, stable, 0.02))
    _report(f"near-180 {fov_name} rotated", counts)


@pytest.mark.parametrize("fov_name", list(NEAR_180))
def test_near_180_double_sources_generic_kernel(torch_cuda, fov_name):
    """Layouts the staged kernels do not take (1, 2 and 4 channels; an odd source width) go
    through remap_generic_kernel: bit-exact on an unrotated output."""
    for width, channels in ((672, 1), (672, 2), (672, 4), (671, 3)):
        sg, og, frames = _near_180_source(NEAR_180[fov_name], width, channels)
        for k, frame in enumerate(frames):
            got = helpers.product_remap(og, (), sg, frame)
            want = numpy_port.remap(og, (), sg, frame)
            assert got.shape == want.shape and np.array_equal(got, want), \
                (fov_name, width, channels, k, mismatch_report(got, want))


@pytest.mark.parametrize("fov_name", list(NEAR_180))
def test_near_180_double_sources_row_bands(torch_cuda, fov_name):
    """batch.remap_row_band through a near-180 double source: tile-aligned bands (staged kernels)
    and odd ones (direct kernel), bit-exact unrotated and on stable pixels rotated."""
    torch = torch_cuda
    from photonbend_b200.batch import remap_row_band, shard_rows

    sg, og, frames = _near_180_source(NEAR_180[fov_name])
    counts = {}
    for rots in ((), ROT):
        cmap = helpers.product_map(og, rots)
        for k, frame in enumerate(frames):
            want = numpy_port.remap(og, rots, sg, frame)
            exact = helpers.stable_pixel_mask(sg, frame, numpy_port.coordinate_map(og, rots)) if rots \
                else np.ones(want.shape[:2], bool)
            dev = torch.from_numpy(frame).cuda()
            source = helpers.product_image(sg, dev)
            bands = [shard_rows(og["height"], r, 3) for r in range(3)] + \
                [range(5, 133), range(0, 1), range(64, 128), range(351, 352), range(170, 183)]
            for rows in bands:
                got = remap_row_band(source, cmap, dev, rows).cpu().numpy()
                sl = slice(rows.start, rows.stop)
                _tally(counts, "rotated" if rots else "unrotated",
                       compare((fov_name, len(rots), k, rows), got, want[sl], exact[sl], 0.02))
    _report(f"near-180 {fov_name} row bands", counts)


@pytest.mark.parametrize("fov_name", list(NEAR_180))
def test_near_180_double_sources_explicit_maps(torch_cuda, fov_name):
    """The explicit-map gather (gather_from_map_kernel) through a near-180 double source, the
    map as an ndarray and as a CUDA tensor, against the oracle sampling the same array."""
    torch = torch_cuda
    sg, og, frames = _near_180_source(NEAR_180[fov_name])
    counts = {}
    for rots in ((), ROT):
        explicit = np.array(helpers.product_map(og, rots))
        for k, frame in enumerate(frames):
            want = numpy_port.sample(sg, frame, explicit.copy())
            exact = stable_mask(sg, frame, explicit) if rots else np.ones(want.shape[:2], bool)
            source = helpers.product_image(sg, frame)
            kind = "rotated" if rots else "unrotated"
            _tally(counts, kind, compare((fov_name, len(rots), k, "ndarray"),
                                         source.process_coordinate_map(explicit.copy()), want, exact, 0.02))
            got_dev = source.process_coordinate_map(torch.from_numpy(explicit.copy()).cuda())
            _tally(counts, kind, compare((fov_name, len(rots), k, "cuda"), got_dev, want, exact, 0.02))
    _report(f"near-180 {fov_name} explicit maps", counts)


# ------------------------------------------------------------------------ edge-value maps

# element bytes -> a dtype of that width (bits are bits: NaN payloads of the image pass through)
WIDE = {2: np.uint16, 4: np.float32, 8: np.float64}


def _source_images(sg, seed):
    """uint8 and every wide pixel shape (2, 4, 8-byte elements x 1..4 channels) of random bits"""
    rng = np.random.default_rng(seed)
    h, w = sg["height"], sg["width"]
    images = [("uint8", rng.integers(0, 256, (h, w, 3), dtype=np.uint8))]
    for e, dt in WIDE.items():
        for c in (1, 2, 3, 4):
            raw = rng.integers(0, 256, (h, w, c * e), dtype=np.uint8)
            images.append((f"{np.dtype(dt).name}x{c}", raw.view(dt).reshape(h, w, c)))
    return images


@pytest.mark.parametrize("src_size", [(40, 80), (27, 51), (48, 96)])
def test_equirect_sources_on_edge_maps_are_bit_exact(torch_cuda, src_size):
    """Equirect sources have no libm on their path (division, truncation, Python-sign modulo):
    every pixel must be the oracle's, for uint8 and all twelve wide pixel shapes, the map passed as
    an ndarray, a CUDA tensor and an edited lazy map, and the caller's map must be left zeroed
    exactly as the reference leaves it."""
    torch = torch_cuda
    sg = {"kind": "equirect", "height": src_size[0], "width": src_size[1]}
    edge = equirect_edge_map(sum(src_size), *src_size)
    images = _source_images(sg, sum(src_size))
    oracle_map = edge.copy()
    numpy_port.sample(sg, images[0][1], oracle_map)  # zeroes the invalid entries in place
    for name, image in images:
        want = numpy_port.sample(sg, image, edge.copy())
        source = helpers.product_image(sg, image)

        host = edge.copy()
        got = source.process_coordinate_map(host)
        assert got.dtype == image.dtype and got.shape == want.shape, name
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (name, "ndarray", mismatch_report(
            got.view(np.uint8), want.view(np.uint8)))
        assert np.array_equal(host.view(np.uint64), oracle_map.view(np.uint64)), (name, "ndarray side effect")

        dev = torch.from_numpy(edge.copy()).cuda()
        got = source.process_coordinate_map(dev)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (name, "cuda")
        assert np.array_equal(dev.cpu().numpy().view(np.uint64), oracle_map.view(np.uint64)), (name, "cuda side effect")

        lazy = helpers.product_image({"kind": "equirect", "height": edge.shape[0], "width": edge.shape[1]},
                                     np.zeros(edge.shape, np.uint8)).get_coordinate_map()
        lazy[...] = edge
        got = source.process_coordinate_map(lazy)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (name, "edited lazy map")
        assert np.array_equal(np.asarray(lazy).view(np.uint64), oracle_map.view(np.uint64)), (name, "lazy side effect")
    assert len(images) == 13
    print(f"equirect {src_size}: {edge.shape[0] * edge.shape[1]} edge entries x 13 pixel shapes x 3 map kinds bit-exact")


CAMERA_SOURCES = [(name, sg) for name, sg in case_matrix.source_geometries() if sg["kind"] == "camera"]


def test_camera_sources_on_edge_maps(torch_cuda):
    """Every built-in lens as a camera source: bit-exact at longitude +-0.0 through an
    equidistant lens, bit-exact on stable pixels everywhere else."""
    torch = torch_cuda
    counts = {}
    lenses = set()
    for i, (name, sg) in enumerate(CAMERA_SOURCES):
        lenses.add(sg["lens"])
        edge = camera_edge_map(100 + i, sg)
        image = case_matrix.case_image(sg, 200 + i)
        want = numpy_port.sample(sg, image, edge.copy())
        exact = stable_mask(sg, image, edge)
        if sg["lens"] == "equidistant":
            exact |= edge[:, :, 1] == 0.0
        source = helpers.product_image(sg, image)
        _tally(counts, "camera", compare((name, "ndarray"), source.process_coordinate_map(edge.copy()), want,
                                         exact, 0.2))
        _tally(counts, "camera", compare((name, "cuda"), source.process_coordinate_map(torch.from_numpy(edge.copy()).cuda()),
                                         want, exact, 0.2))
    assert lenses == set(case_matrix.LENSES)
    _report("edge maps", counts)


@pytest.mark.parametrize("fov_name", ["195", "180.00000000001", "179.99999999999"])
def test_double_sources_on_edge_maps(torch_cuda, fov_name):
    """Double sources (every lens a double image takes) on maps aimed at the blend band's edges:
    bit-exact at longitude +-0.0 through an equidistant lens, bit-exact on stable pixels
    everywhere else."""
    torch = torch_cuda
    fov = rad(float(fov_name))
    counts = {}
    for i, lens in enumerate(("equidistant", "equisolid", "orthographic", "stereographic", "thoby")):
        sg = {"kind": "double", "height": 40, "width": 80, "lens": lens, "fov": fov}
        edge = double_edge_map(300 + i, sg)
        image = case_matrix.case_image(sg, 400 + i)
        want = numpy_port.sample(sg, image, edge.copy())
        exact = stable_mask(sg, image, edge)
        if lens == "equidistant":
            exact |= edge[:, :, 1] == 0.0
        source = helpers.product_image(sg, image)
        _tally(counts, "double", compare((fov_name, lens, "ndarray"), source.process_coordinate_map(edge.copy()),
                                         want, exact, 0.25))
        _tally(counts, "double", compare((fov_name, lens, "cuda"),
                                         source.process_coordinate_map(torch.from_numpy(edge.copy()).cuda()),
                                         want, exact, 0.25))
    _report(f"edge maps, sensor fov {fov_name}", counts)


def test_rotate_coordinate_map_on_edge_maps(torch_cuda):
    """Rotation.rotate_coordinate_map (rotate_map_kernel) on an edge map, as an ndarray and as a
    CUDA tensor: flags and NaN positions as the oracle's, the caller's map zeroed bit for bit as the
    reference zeroes it, finite values within 1e-9; then sampled through an equirect source."""
    torch = torch_cuda
    from photonbend_b200.core.rotation import Rotation

    sg = {"kind": "equirect", "height": 40, "width": 80}
    image = case_matrix.case_image(sg, 31)
    edge = equirect_edge_map(5, 40, 80)
    oracle_in = edge.copy()
    want = numpy_port.rotate_map(oracle_in, numpy_port.rotation_matrix(*ROT[0]))
    rot = Rotation(*ROT[0])
    assert np.array_equal(rot.rotation_matrix, numpy_port.rotation_matrix(*ROT[0]))
    host = edge.copy()
    dev = torch.from_numpy(edge.copy()).cuda()
    got_dev = rot.rotate_coordinate_map(dev).cpu().numpy()
    results = {"ndarray": (rot.rotate_coordinate_map(host), host), "cuda": (got_dev, dev.cpu().numpy())}
    counts = {}
    for kind, (got, caller) in results.items():
        assert np.array_equal(caller.view(np.uint64), oracle_in.view(np.uint64)), kind
        assert np.array_equal(got[:, :, 2].view(np.uint64), want[:, :, 2].view(np.uint64)), kind
        assert np.array_equal(np.isnan(got), np.isnan(want)), kind
        finite = np.isfinite(want[:, :, 0]) & np.isfinite(want[:, :, 1])
        assert np.array_equal(finite, np.isfinite(got[:, :, 0]) & np.isfinite(got[:, :, 1])), kind
        assert np.all(np.abs(got[:, :, 0] - want[:, :, 0])[finite] < 1e-9), kind
        gx, gz = np.sin(got[:, :, 0]) * np.cos(got[:, :, 1]), np.sin(got[:, :, 0]) * np.sin(got[:, :, 1])
        wx, wz = np.sin(want[:, :, 0]) * np.cos(want[:, :, 1]), np.sin(want[:, :, 0]) * np.sin(want[:, :, 1])
        assert np.all(np.hypot(gx - wx, gz - wz)[finite] < 1e-9), kind
        picked = numpy_port.sample(sg, image, want.copy())
        sampled = helpers.product_image(sg, image).process_coordinate_map(got.copy())
        _tally(counts, "rotated equirect", compare(kind, sampled, picked, stable_mask(sg, image, want), 0.02))
    _report("edge maps", counts)


def _map_projection_cases(seed):
    """Edge maps for map_projection, each with the property named by its key."""
    rng = np.random.default_rng(seed)
    shape = (160, 224)
    base = equirect_edge_map(seed, 40, 80, shape)
    c = 255.0 / (np.pi * 2)  # the scale of the longitude channel, projection.py:583-584
    ks = np.arange(-3, 300)
    halves = _around((ks + 0.5) / c, 2)
    halves = halves[np.mod(c * halves, 1.0) == 0.5]  # scaled value exactly k + .5
    assert halves.size > 100
    near_256 = _around(np.array([255.5, 256.0, 256.5, -0.5, -255.5]) / c, 3)
    lon = _pick(rng, [halves, near_256, _huge(1 / c), rng.uniform(-10, 10, 64), SPECIALS], shape)
    flags = _flags(rng, shape)
    valid = np.argwhere(flags == 0)
    cases = {"finite": _stack(rng.uniform(0, 3, shape), lon, flags)}

    def edited(channel, value, *entries):
        m = cases["finite"].copy()
        for k in entries:
            m[valid[k][0], valid[k][1], channel] = value
        return m

    cases["one NaN latitude"] = edited(0, np.nan, 7)
    cases["+inf latitude"] = edited(0, np.inf, 11)
    cases["-inf latitude"] = edited(0, -np.inf, 11)
    m = cases["finite"].copy()
    m[:, :, 0] = np.where(flags == 0, 0.7, m[:, :, 0])
    cases["all valid latitudes equal"] = m
    m = cases["finite"].copy()
    m[:, :, 2] = np.where(flags == 0, 1.0, flags)
    m[valid[3][0], valid[3][1], 2] = -0.0
    cases["one valid entry"] = m
    # lo = 0, hi = 255: factor 1, so the red channel rounds latitudes of k + .5 (and their
    # neighbours) as they are
    lat = _pick(rng, [_around(np.arange(0, 255) + 0.5, 1), np.arange(0, 256.0)], shape)
    lat[0, 0], lat[0, 1] = 0.0, 255.0
    m = _stack(lat, lon, flags)
    m[0, 0, 2] = m[0, 1, 2] = 0.0
    cases["latitudes on .5"] = m
    cases["edge latitudes"] = base  # NaN, inf and huge latitudes among the valid ones
    return cases


def test_map_projection_on_edge_maps_is_bit_exact(torch_cuda):
    """map_projection (map_range_kernel + map_projection_kernel) has no libm: rint is NumPy's
    half-to-even and cast_u8 its uint8 cast, so every pixel and the zeroing of the caller's map
    must be the oracle's, for an ndarray and a CUDA tensor."""
    torch = torch_cuda
    from photonbend_b200.core.projection import map_projection

    for name, m in _map_projection_cases(17).items():
        oracle_map = m.copy()
        with np.errstate(all="ignore"):
            want = numpy_port.map_projection(oracle_map)
        host = m.copy()
        got = map_projection(host)
        assert np.array_equal(got, want), (name, "ndarray", mismatch_report(got, want))
        assert np.array_equal(host.view(np.uint64), oracle_map.view(np.uint64)), (name, "ndarray side effect")
        dev = torch.from_numpy(m.copy()).cuda()
        got = map_projection(dev)
        assert np.array_equal(got, want), (name, "cuda", mismatch_report(got, want))
        assert np.array_equal(dev.cpu().numpy().view(np.uint64), oracle_map.view(np.uint64)), (name, "cuda side effect")
