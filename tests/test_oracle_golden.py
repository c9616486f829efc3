"""Pins the CPU oracles (oracle/) to golden vectors produced by the LIVE reference
(tests/golden/make_golden.py).  CPU only.

* oracle/numpy_port.py must be bit-identical: every output image hash and every float64
  coordinate-map hash of the 1.7k-case matrix must match.
* oracle/pb_oracle.c (glibc libm instead of NumPy's SIMD kernels) must match every stored
  output except for the one legitimate class of difference SURVEY.md section 7 describes: a 1-LSB
  change of the float64 blend of a *rotated double-fisheye source*.
"""

import hashlib
import json
import os
import platform

import numpy as np
import pytest

import case_matrix
from conftest import GOLDEN, mismatch_report
from oracle import c_port, numpy_port


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


CASES = case_matrix.all_cases()


def test_matrix_is_the_one_the_goldens_were_made_from(golden_small):
    meta, _, _ = golden_small
    assert all(cid in meta for cid, *_ in CASES)
    assert len(CASES) > 1500


def test_numpy_port_bit_identical_to_reference(golden_small):
    meta, _, _ = golden_small
    for cid, og, rots, sg, seed in CASES:
        image = case_matrix.case_image(sg, seed)
        cmap = numpy_port.coordinate_map(og, rots)
        final_map = cmap.copy()
        out = numpy_port.sample(sg, image, cmap)
        assert _sha(out) == meta[cid]["out_sha256"], cid
        assert _sha(final_map) == meta[cid]["map_sha256"], cid


def test_numpy_port_channel_layouts(golden_small):
    meta, outputs, _ = golden_small
    extra = [k for k in meta if k.endswith("__grey") or k.endswith("__rgba")]
    assert extra
    by_id = {c[0]: c for c in CASES}
    for key in extra:
        cid, tag = key.rsplit("__", 1)
        _, og, rots, sg, seed = by_id[cid]
        image = case_matrix.case_image(sg, seed, meta[key]["channels"])
        out = numpy_port.remap(og, rots, sg, image)
        assert np.array_equal(out, outputs[key]), key


def test_numpy_port_row_bands_equal_whole(golden_small):
    _, outputs, _ = golden_small
    by_id = {c[0]: c for c in CASES}
    for cid in list(outputs.files)[::40]:
        if cid not in by_id:
            continue
        _, og, rots, sg, seed = by_id[cid]
        image = case_matrix.case_image(sg, seed)
        h = outputs[cid].shape[0]
        bands = [numpy_port.remap(og, rots, sg, image, rows=(a, b))
                 for a, b in ((0, h // 3), (h // 3, h - 2), (h - 2, h))]
        assert np.array_equal(np.concatenate(bands, 0), outputs[cid]), cid


def test_c_port_matches_reference_outputs(golden_small):
    meta, outputs, _ = golden_small
    by_id = {c[0]: c for c in CASES}
    n_checked = n_lsb = 0
    for cid in outputs.files:
        if cid not in by_id:
            continue
        _, og, rots, sg, seed = by_id[cid]
        image = case_matrix.case_image(sg, seed)
        got = c_port.remap(og, rots, sg, image, threads=1)
        want = outputs[cid]
        n_checked += 1
        if np.array_equal(got, want):
            continue
        exact, max_abs, n_bad = mismatch_report(got, want)
        # only a rotated double-fisheye source may differ, by one pixel, by one LSB
        assert sg["kind"] == "double" and len(rots) > 0, cid
        assert max_abs == 1 and n_bad <= 2, (cid, max_abs, n_bad)
        n_lsb += 1
    assert n_checked > 400
    assert n_lsb <= n_checked // 50


def test_c_port_coordinate_maps_close_to_reference(golden_small):
    _, _, maps = golden_small
    geoms = dict(case_matrix.output_geometries())
    rots = dict(case_matrix.ROTATION_SETS)
    for key in maps.files:
        oname, rname = key.split("__")
        want = maps[key]
        got = c_port.coordinate_map(geoms[oname], rots[rname], threads=1)
        assert got.shape == want.shape
        assert np.array_equal(got[:, :, 2] != 0, want[:, :, 2] != 0), key
        valid = want[:, :, 2] == 0
        both_nan = np.isnan(got) & np.isnan(want)
        # longitude is meaningless (and ill-conditioned) at the poles: compare it through the ray direction
        err_lat = np.abs(got[:, :, 0] - want[:, :, 0])
        assert np.all((err_lat < 1e-9) | both_nan[:, :, 0] | ~valid), key
        gx, gz = np.sin(got[:, :, 0]) * np.cos(got[:, :, 1]), np.sin(got[:, :, 0]) * np.sin(got[:, :, 1])
        wx, wz = np.sin(want[:, :, 0]) * np.cos(want[:, :, 1]), np.sin(want[:, :, 0]) * np.sin(want[:, :, 1])
        err_dir = np.hypot(gx - wx, gz - wz)
        assert np.all((err_dir < 1e-9) | both_nan[:, :, 0] | both_nan[:, :, 1] | ~valid), key
        if rname == "r0":  # no libm-dependent rotation: unrotated maps are bit-identical
            if geoms[oname]["kind"] == "equirect" or geoms[oname]["lens"] == "equidistant":
                assert np.array_equal(got, want, equal_nan=True), key


def test_c_port_threads_equal_single_thread():
    cid, og, rots, sg, seed = CASES[len(CASES) // 2]
    og = dict(og, height=og["height"] * 4, width=og["width"] * 4)
    image = case_matrix.case_image(sg, seed)
    a = c_port.remap(og, rots, sg, image, threads=1)
    b = c_port.remap(og, rots, sg, image, threads=4)
    c = c_port.remap(og, rots, sg, image, rows=(5, 17), threads=2)
    assert np.array_equal(a, b)
    assert np.array_equal(a[5:17], c)


def numpy_u8_cast_model(v):
    """NumPy's float64 -> uint8 cast on x86-64, as the kernels (cast_u8 in csrc/pb_device.cuh) and
    pb_oracle.c restate it: truncation to a 32-bit integer (cvttsd2si), low byte kept; NaN and
    |v| >= 2^31 become INT32_MIN, whose low byte is 0."""
    v = np.asarray(v, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        fits = np.abs(v) < 2.0**31
    t = np.where(fits, np.trunc(np.where(fits, v, 0.0)), -(2.0**31)).astype(np.int64)
    return (t & 0xFF).astype(np.uint8)


@pytest.mark.skipif(platform.machine().lower() not in ("x86_64", "amd64"),
                    reason="the kernels restate NumPy's x86-64 cast; other hosts saturate")
def test_numpy_uint8_cast_is_the_32_bit_truncation_the_kernels_restate():
    """ndarray.astype(np.uint8) of float64 on this host against numpy_u8_cast_model, over the
    values where 8-, 32- and 64-bit truncations part ways, contiguous, strided and 3-D."""
    tiny = np.finfo(np.float64).smallest_subnormal
    edges = [np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, tiny, -tiny, 1e-310, -1e-310,
             0.5, -0.5, 0.999999, -0.999999, 1.5, -1.5, 255.0, 255.5, 255.9999999, 256.0, 256.5,
             -255.9999, -256.0, -256.5, 300.7, -300.7, 2.0**63, -(2.0**63), 2.0**64, 1e300, -1e300]
    for base in (2.0**31, 2.0**32, 2.0**52, 2.0**53):
        for d in (-7.0, -1.0, -0.5, 0.0, 0.5, 1.0, 7.0):
            edges += [base + d, -(base + d)]
        edges += [np.nextafter(base, 0), np.nextafter(base, np.inf), -np.nextafter(base, 0), -np.nextafter(base, np.inf)]
    edges = np.array(edges, dtype=np.float64)
    want = numpy_u8_cast_model(edges)
    assert want[np.isnan(edges)].tolist() == [0, 0]
    assert numpy_u8_cast_model([2.0**31 + 7, 300.7, -1.5, 255.9999999, -256.5]).tolist() == [0, 44, 255, 255, 0]
    rng = np.random.default_rng(31)
    mags = 10.0 ** rng.uniform(-323, 308, 200_000)
    sweep = np.concatenate([edges, mags * rng.choice([-1.0, 1.0], mags.size),
                            rng.uniform(-2.0**33, 2.0**33, 100_000), rng.uniform(-600, 600, 100_000)])
    with np.errstate(invalid="ignore"):
        assert np.array_equal(sweep.astype(np.uint8), numpy_u8_cast_model(sweep))
        assert np.array_equal(np.repeat(sweep, 2)[1::2].astype(np.uint8), numpy_u8_cast_model(sweep))
        cube = sweep[: (sweep.size // 60) * 60].reshape(-1, 20, 3)
        assert np.array_equal(cube.astype(np.uint8), numpy_u8_cast_model(cube))
        assert np.array_equal(cube[:, ::2, 1:].astype(np.uint8), numpy_u8_cast_model(cube[:, ::2, 1:]))


# Double-fisheye sensor fovs within 1e-9 rad of pi: the blend band 2 * (fov/2 - pi/2) nearly
# vanishes and its weights reach 1e7 .. 1e13, beyond the 32 bits of NumPy's uint8 cast.
NEAR_180_FOVS = {
    "nextafter_up": float(np.nextafter(np.pi, np.inf)),
    "nextafter_down": float(np.nextafter(np.pi, 0.0)),
    "pi_plus_1e-12": np.pi + 1e-12,
    "pi_minus_1e-12": np.pi - 1e-12,
    "180.000000001": case_matrix.rad(180.000000001),
    "180.00000000001": case_matrix.rad(180.00000000001),
    "179.99999999999": case_matrix.rad(179.99999999999),
    "pi": np.pi,
    "180.0000001": case_matrix.rad(180.0000001),
}


@pytest.mark.parametrize("fov_name", list(NEAR_180_FOVS))
def test_c_port_blend_of_near_180_degree_double_sources(fov_name):
    """oracle/pb_oracle.c against the NumPy oracle (bit-identical to the reference) on double
    sources whose blend weights overflow int32: the C oracle has to cast the blend to uint8 the
    way NumPy does, or every pixel of the band rows differs."""
    fov = NEAR_180_FOVS[fov_name]
    for (h, w), og in (((336, 672), {"kind": "equirect", "height": 352, "width": 704}),
                       ((200, 400), {"kind": "equirect", "height": 400, "width": 800})):
        sg = {"kind": "double", "height": h, "width": w, "lens": "equidistant", "fov": fov}
        for image in (np.full((h, w, 3), 200, np.uint8), case_matrix.case_image(sg, 7)):
            for rots in ((), ((0.3, -0.7, 1.1),)):
                got = c_port.remap(og, rots, sg, image)
                want = numpy_port.remap(og, rots, sg, image)
                assert np.array_equal(got, want), (fov_name, h, len(rots), mismatch_report(got, want))


@pytest.mark.parametrize("bad_fov_deg", [179.0, 180.0])
def test_rectilinear_fov_limit_raises_like_reference(bad_fov_deg):
    # reference lens.py:88-94 via projection.py:141-144
    geom = {"kind": "camera", "height": 8, "width": 8, "lens": "rectilinear",
            "fov": case_matrix.rad(bad_fov_deg), "magnitude": 3.5}
    with pytest.raises(ValueError):
        numpy_port.focal_distance(geom)


def test_tiny_and_degenerate_sizes_against_the_reference():
    """One-pixel / one-row images, odd double widths, non-2:1 panoramas (tests/tiny_matrix.py):
    both oracles against outputs of the live reference (tests/golden/make_golden_tiny.py)."""
    import tiny_matrix
    from oracle import c_port, numpy_port

    with open(os.path.join(GOLDEN, "tiny_cases.json")) as fh:
        meta = json.load(fh)
    outputs = np.load(os.path.join(GOLDEN, "tiny_outputs.npz"))
    n = n_c_diff = 0
    for cid, og, rots, sg, seed in tiny_matrix.all_cases():
        assert "raises" not in meta[cid]
        image = tiny_matrix.case_image(sg, seed)
        want = outputs[cid]
        got = numpy_port.remap(og, rots, sg, image)
        assert got.shape == want.shape and np.array_equal(got, want), cid
        got_c = c_port.remap(og, rots, sg, image)
        assert got_c.shape == want.shape
        n_c_diff += int((got_c != want).any(axis=2).sum())  # glibc libm vs NumPy's SIMD kernels
        n += 1
    assert n == 180 and n_c_diff <= 4, n_c_diff


def test_degenerate_case_census():
    """How many cases of the small matrix have MORE than 1 % of the reference's own pixels hanging
    on the last ulps of NumPy's libm (helpers.stable_pixel_mask; e.g. an un-rotated map onto an
    equirect source puts pixel centres exactly on row boundaries, a 360-degree stereographic lens
    has an infinite image radius).  Counted with the oracle alone; tests/test_gpu_parity.py may
    treat at most this many cases as "degenerate" (stable pixels only), so the constants there
    are pinned here."""
    import helpers
    import test_gpu_parity as gpu_tests
    from oracle import numpy_port

    by_id = {c[0]: c for c in case_matrix.all_cases()}

    def degenerate(cid, channels=3):
        _, og, rots, sg, seed = by_id[cid]
        image = case_matrix.case_image(sg, seed, channels)
        try:
            cmap = numpy_port.coordinate_map(og, rots)
        except ValueError:
            return False
        return bool((~helpers.stable_pixel_mask(sg, image, cmap)).mean() > 0.01)

    assert sum(degenerate(cid) for cid in by_id) == gpu_tests.MAX_DEGENERATE_MATRIX
    with open(os.path.join(GOLDEN, "small_cases.json")) as fh:
        meta = json.load(fh)
    outputs = np.load(os.path.join(GOLDEN, "small_outputs.npz"))
    n = sum(degenerate("__".join(key.split("__")[:3]), meta[key].get("channels", 3)) for key in outputs.files)
    assert n == gpu_tests.MAX_DEGENERATE_GOLDEN


def test_c_port_config5_frames_at_full_size():
    """oracle/pb_oracle.c on frames of BASELINE config 5 (seeds 1234 + k, 3840x7680 double fisheye
    -> 3840x7680 equirect): sha256-identical to the live reference's outputs
    (tests/golden/cfg5_frames.json) -- the checker bench.py's ``parity`` block uses."""
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["cfg5"]
    with open(os.path.join(GOLDEN, "cfg5_frames.json")) as fh:
        golden = json.load(fh)["frames"]
    assert len(golden) >= 8
    for k in (0, 3, 7):
        image = workloads.source_image(wl, frame=k)
        assert _sha(image) == golden[k]["src_sha256"]
        assert _sha(c_port.remap(wl["out"], wl["rotations"], wl["src"], image)) == golden[k]["out_sha256"], k


def test_numpy_port_map_projection_matches_the_reference(golden_small):
    """oracle.numpy_port.map_projection vs the live reference's map_projection outputs
    (tests/golden/map_projection.npz, made by make_golden_mapproj.py), incl. the in-place zeroing."""
    _, _, maps = golden_small
    golden = np.load(os.path.join(GOLDEN, "map_projection.npz"))
    assert len(golden.files) >= 20
    for key in golden.files:
        cmap = maps[key].copy()
        assert np.array_equal(numpy_port.map_projection(cmap), golden[key]), key
        invalid = cmap[:, :, 2] != 0
        assert np.all(cmap[invalid, :2] == 0)
