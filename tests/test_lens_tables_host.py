"""User-defined lenses on the host: the table oracle's interpolation (tests/table_oracle.py) against a
direct evaluation, the ranges the product samples a user lens on (core/projection.py:
_custom_lens_table), and the distance between the table oracle and the reference's own evaluation of
the user's callables, as a bound derived from the table's spacing instead of a pixel count."""

import warnings

import numpy as np
import pytest

import table_oracle
from oracle import numpy_port

rad = np.deg2rad


def _direct(table, x_max, x):
    """lens_table_at of pb_device.cuh, one Python float at a time"""
    n = len(table)
    scale = (n - 1) / x_max
    if x != x:
        return x
    t = x * scale
    t = 0.0 if t < 0.0 else t
    i = n - 2 if t >= n - 1 else int(t)
    fr = min(t - i, 1.0)
    a, b = float(table[i]), float(table[i + 1])
    return a + (b - a) * fr


@pytest.mark.parametrize("n", [2, 3, 17, 1025, 65537])
def test_table_at_is_the_kernels_interpolation(n):
    rng = np.random.default_rng(n)
    x_max = float(rng.uniform(0.5, 4.0))
    xs = np.linspace(0.0, x_max, n)
    table = np.sin(3 * xs) + 0.5 * xs
    k = np.arange(n)
    mid = (xs[:-1] + xs[1:]) / 2
    probes = np.concatenate([xs, mid, rng.uniform(-1.0, 2 * x_max, 4000), [-0.0, -1e300, x_max, np.nextafter(x_max, 9),
                                                                               2 * x_max, 1e300, np.inf, -np.inf, np.nan]])
    got = table_oracle.table_at(table, x_max, probes)
    want = np.array([_direct(table, x_max, float(x)) for x in probes])
    assert np.array_equal(got, want, equal_nan=True)
    assert np.array_equal(np.signbit(got), np.signbit(want))
    # at the samples: the sample itself (to the rounding of x * scale)
    at = table_oracle.table_at(table, x_max, xs)
    step = np.abs(np.diff(table)).max()
    assert np.allclose(at, table[k], rtol=0, atol=4e-16 * (step + np.abs(table).max()) * 4)
    # at midpoints: the mean of the two samples
    assert np.allclose(table_oracle.table_at(table, x_max, mid), (table[:-1] + table[1:]) / 2, rtol=0, atol=1e-14)
    # beyond x_max (and at inf): the last interval's end, i.e. the last sample; below 0: the first
    last = table[-2] + (table[-1] - table[-2])
    assert np.all(table_oracle.table_at(table, x_max, np.array([x_max * 1.5, 1e300, np.inf])) == last)
    assert np.all(table_oracle.table_at(table, x_max, np.array([-1.0, -np.inf, -0.0])) == table[0])
    assert np.isnan(table_oracle.table_at(table, x_max, np.array([np.nan]))).all()
    # a table with NaN / inf samples spreads them to its two intervals only
    bad = table.copy()
    bad[n // 2] = np.nan
    got = table_oracle.table_at(bad, x_max, probes)
    want = np.array([_direct(bad, x_max, float(x)) for x in probes])
    assert np.array_equal(got, want, equal_nan=True)


def test_table_at_with_two_samples_is_a_clamped_line():
    x = np.linspace(-1.0, 3.0, 401)
    got = table_oracle.table_at(np.array([1.0, 5.0]), 2.0, x)
    assert np.allclose(got, 1.0 + 2.0 * np.clip(x, 0.0, 2.0), rtol=0, atol=1e-15)


# ------------------------------------------------------------------------------------ ranges


def _kb_lens():
    from photonbend_b200.core.lens import Lens

    return Lens(lambda t: t * (1 + 0.08 * t**2 + 0.01 * t**4), lambda r: r / (1 + 0.08 * r**2))


@pytest.mark.parametrize("kind,h,w,mag", [("camera", 170, 336, 150.5), ("camera", 171, 337, None),
                                          ("camera", 64, 301, 20.25), ("double", 170, 336, None),
                                          ("double", 171, 339, None), ("double", 96, 194, None)])
def test_output_table_covers_every_pixel_radius(kind, h, w, mag):
    """The reverse table of an output spans the largest radius its rays evaluate (double outputs:
    of a width // 2 half), so no output pixel reads the clamp; a source samples [0, pi]."""
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage

    lens = _kb_lens()
    arr = np.zeros((h, w, 3), np.uint8)
    image = (CameraImage(arr, rad(190), lens, magnitude=mag) if kind == "camera" else
             DoubleCameraImage(arr, rad(195), lens))
    out, src = image._output_geometry(), image._source_geometry()
    assert src.table_max == np.pi and src.table.size == out.table.size
    seen = []

    def reverse(d):
        seen.append(float(np.nanmax(d)))
        return lens.reverse_function(d)

    geom = table_oracle.geom_of(image)
    geom["lens"] = table_oracle.TableLens(lens.forward_function, reverse, per_pixel="callable")
    with table_oracle.patched(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        numpy_port.output_rays(geom)
    d_max = max(seen)
    assert d_max <= out.table_max <= d_max * (1 + 1e-8) + 1e-11, (d_max, out.table_max)
    n = out.table.size
    assert d_max * ((n - 1) / out.table_max) <= n - 1


# ------------------------------------------------------------------------------------ table vs callables

LENSES = {
    "equisolid": (lambda t: 2 * np.sin(t / 2), lambda r: 2 * np.arcsin(r / 2), lambda t: 0.5 * np.abs(np.sin(t / 2))),
    "kannala-brandt": (lambda t: t * (1 + 0.08 * t**2 + 0.01 * t**4), lambda r: r / (1 + 0.08 * r**2),
                       lambda t: np.abs(0.48 * t + 0.2 * t**3)),
    "wavy": (lambda t: t + 0.05 * np.sin(6 * t), lambda r: r - 0.05 * np.sin(6 * r),
             lambda t: np.abs(1.8 * np.sin(6 * t))),
}


def _second_derivative_max(f2, lo, hi):
    xs = np.linspace(lo, hi, 20001)
    return float(np.max(f2(xs)))


def _interval_m2(fn, x_max, n):
    """max |f''| over each interval [x_i, x_i+1] of a table of n samples on [0, x_max], from second
    divided differences on a grid 8 times finer (NaN where f is not finite there)"""
    k = 8
    xs = np.linspace(0.0, x_max, k * (n - 1) + 1)
    step = xs[1] - xs[0]
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        f = np.asarray(fn(xs), dtype=np.float64)
    d2 = np.abs(f[2:] - 2 * f[1:-1] + f[:-2]) / (step * step)
    d2 = np.concatenate([d2[:1], d2, d2[-1:]])  # per fine point
    return np.max(np.lib.stride_tricks.sliding_window_view(d2, k + 1)[::k], axis=1)


def _radii(og):
    """radius in focal units of each output pixel (camera_rays / double_rays)"""
    h, w = og["height"], og["width"]
    n_cols = w // 2 if og["kind"] == "double" else w
    xs = np.linspace(-n_cols / 2 + 0.5, n_cols / 2 - 0.5, num=n_cols)
    if og["kind"] == "double":
        xs = np.concatenate([xs, xs * (-1)], 0)
    ys = np.linspace(h / 2 - 0.5, -h / 2 + 0.5, num=h)
    gy, gx = np.meshgrid(ys, xs, sparse=True, indexing="ij")
    return np.sqrt(gx**2 + gy**2) / numpy_port.focal_distance(og)


def moved_any(cmap_t, cmap_c, seg_h, seg_w, w):
    """pixels whose truncated panorama row or column differs between two maps"""
    with np.errstate(all="ignore"):
        rows = [np.trunc(c[:, :, 0] / seg_h) for c in (cmap_t, cmap_c)]
        cols = [np.trunc(c[:, :, 1] / seg_w + w / 2) for c in (cmap_t, cmap_c)]
    return ~((rows[0] == rows[1]) & (cols[0] == cols[1]))


def _coords(sg, cmap):
    """[(x, y, r, f)] of each lens a source reads along cmap (a double source: left, then right), unrounded"""
    lat, lon = cmap[:, :, 0], cmap[:, :, 1]
    h, w = sg["height"], sg["width"]
    halves = [(lat, w)] if sg["kind"] == "camera" else [(lat, w // 2), ((lat * -1) + np.pi, w - w // 2)]
    out = []
    for lat_k, wk in halves:
        sub = dict(sg, kind="camera", width=wk, magnitude=sg.get("magnitude"))
        f = numpy_port.focal_distance(sub)
        with np.errstate(all="ignore"):
            r = numpy_port.lens_forward(sg["lens"], lat_k) * f
            p = np.exp(lon * 1j) * r
            out.append((p.real + (wk / 2 - 0.5), (p.imag * (-1)) + (h / 2 - 0.5), r, f))
    return out


@pytest.mark.parametrize("lens", list(LENSES))
@pytest.mark.parametrize("side", ["source", "output"])
def test_table_follows_the_callables_to_a_derived_bound(lens, side):
    """With the default 65537 samples, the table oracle and the callables' oracle pick different
    source pixels only where a coordinate straddles an integer, each by one pixel, and the lens
    values differ by at most h^2 / 8 * max|f''| (h the sample spacing) plus a few ulps -- the
    interpolation error DESIGN section 1 quotes as ~1e-7 px."""
    from photonbend_b200.core.lens import Lens
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, PanoramaImage

    fwd, rev, f2 = LENSES[lens]
    user = Lens(fwd, rev)
    rng = np.random.default_rng(3)
    cases = []
    if side == "source":
        pano = PanoramaImage(np.zeros((160, 320, 3), np.uint8))
        for image in (CameraImage(np.zeros((240, 256, 3), np.uint8), rad(200), user, magnitude=119.5),
                      DoubleCameraImage(np.zeros((192, 384, 3), np.uint8), rad(195), user)):
            for rots in ((), ((0.3, -0.2, 1.0),)):
                cases.append((pano, rots, image))
    else:
        src = PanoramaImage(np.zeros((192, 384, 3), np.uint8))
        for image in (CameraImage(np.zeros((170, 336, 3), np.uint8), rad(170), user, magnitude=150.5),
                      DoubleCameraImage(np.zeros((170, 337, 3), np.uint8), rad(195), user)):
            for rots in ((), ((0.3, -0.2, 1.0),)):
                cases.append((image, rots, src))
    n_diff = 0
    for og_image, rots, sg_image in cases:
        og_t, sg_t = table_oracle.geom_of(og_image), table_oracle.geom_of(sg_image)
        og_c, sg_c = table_oracle.geom_of(og_image, "callable"), table_oracle.geom_of(sg_image, "callable")
        with table_oracle.patched(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if side == "output":
                lat_t = numpy_port.output_rays(og_t)[:, :, 0]
                lat_c = numpy_port.output_rays(og_c)[:, :, 0]
                table = og_image._output_geometry()
                h = table.table_max / (table.table.size - 1)
                # max|g''| of the interval each radius falls in (equisolid: g'' grows without bound
                # towards r = 2, where its domain ends and the table's samples turn NaN)
                m2 = _interval_m2(rev, table.table_max, table.table.size)
                d = _radii(og_t)
                idx = np.minimum((d / h).astype(np.int64), m2.size - 1)
                ok = np.isfinite(lat_t) & np.isfinite(lat_c)
                bound = h * h / 8 * m2[idx] * 1.5 + 4 * np.spacing(np.pi)
                assert np.all(np.abs(lat_t - lat_c)[ok] <= bound[ok]), float(np.max(np.abs(lat_t - lat_c)[ok]))
                # NaN only where the callable itself is NaN or the interval reaches a NaN sample
                nan_sample = ~np.isfinite(table.table[idx]) | ~np.isfinite(table.table[idx + 1])
                assert np.array_equal(np.isnan(lat_t), np.isnan(lat_c) | nan_sample)
            cmap_t = numpy_port.coordinate_map(og_t, rots)
            cmap_c = numpy_port.coordinate_map(og_c, rots)
            img = rng.integers(0, 256, (sg_t["height"], sg_t["width"], 3), dtype=np.uint8)
            got_t = numpy_port.sample(sg_t, img, cmap_t.copy())
            got_c = numpy_port.sample(sg_c, img, cmap_c.copy())
            diff = (got_t != got_c).any(axis=2)
            n_diff += int(diff.sum())
            if side == "source":
                table = sg_image._source_geometry()
                h = table.table_max / (table.table.size - 1)
                pairs = zip(_coords(sg_t, cmap_t), _coords(sg_c, cmap_c))
                for (xt, yt, rt, f), (xc, yc, rc, _) in pairs:
                    inside = ((cmap_t[:, :, 2] == 0) & (xc > -1) & (xc < sg_t["width"] + 1) & (yc > -1) &
                              (yc < sg_t["height"] + 1))
                    bound = h * h / 8 * _second_derivative_max(f2, 0.0, np.pi) * f
                    dr = np.abs(rt - rc)
                    assert np.all(dr[inside] <= bound * 1.01 + 8 * np.spacing(np.abs(rc[inside]))), \
                        (float(np.max(dr[inside])), bound)
                    for a, b in ((xt, xc), (yt, yc)):
                        moved = inside & (np.trunc(a) != np.trunc(b))
                        # a pixel changes only where an integer lies between the two coordinates, one step away
                        assert np.all(np.abs(np.trunc(a[moved]) - np.trunc(b[moved])) == 1)
                        assert np.all(np.floor(np.maximum(a[moved], b[moved])) > np.minimum(a[moved], b[moved]))
                        assert np.all(np.abs(a[moved] - b[moved]) < 1e-5)
            else:  # the panorama's row and column coordinates (numpy_port.sample_equirect)
                seg_h, seg_w = np.pi / sg_t["height"], np.pi / (sg_t["width"] / 2)
                valid = (cmap_t[:, :, 2] == 0) & (cmap_c[:, :, 2] == 0)
                for a, b in ((cmap_t[:, :, 0] / seg_h, cmap_c[:, :, 0] / seg_h),
                             (cmap_t[:, :, 1] / seg_w + sg_t["width"] / 2, cmap_c[:, :, 1] / seg_w + sg_t["width"] / 2)):
                    moved = valid & np.isfinite(a) & np.isfinite(b) & (np.trunc(a) != np.trunc(b))
                    assert np.all(np.abs(np.trunc(a[moved]) - np.trunc(b[moved])) == 1)
                    assert np.all(np.abs(a[moved] - b[moved]) < 1e-3)
                assert not (diff & valid & ~moved_any(cmap_t, cmap_c, seg_h, seg_w, sg_t["width"])).any()
    print(f"{lens} ({side}): {n_diff} pixels differ between the table oracle and the callables")


def test_sample_counts_reach_the_oracle_through_the_python_api(monkeypatch):
    """Tests pick a table length by patching core.projection.lens_table (LENS_TABLE_SAMPLES is bound
    as a default argument): the geometry, its digest and the oracle all see the patched table."""
    import functools

    from photonbend_b200.core import projection
    from photonbend_b200.core.lens import Lens, lens_table

    monkeypatch.setattr(projection, "lens_table", functools.partial(lens_table, samples=17))
    image = projection.CameraImage(np.zeros((40, 48, 3), np.uint8), rad(180), Lens(*LENSES["wavy"][:2]))
    src, out = image._source_geometry(), image._output_geometry()
    assert src.table.size == out.table.size == 17 and src.table_key != out.table_key
    geom = table_oracle.geom_of(image)
    assert geom["lens"].source[0] is src.table and geom["lens"].output[0] is out.table
    assert np.array_equal(src.table, LENSES["wavy"][0](np.linspace(0, np.pi, 17)))
