"""Parity of the CUDA path (through the C ABI, libpbremap.so) with the reference.  GPU only.

Bar (BASELINE.json): >= 99.99 % of output pixels bit-exact with the reference's CPU result, and
every differing pixel attributed to (a) a +-1 source-index flip at an integer boundary or (b) the
1-LSB truncation of the float64 blend of a double-fisheye source.  The checker is the oracle
(oracle/numpy_port.py bit-identical to the reference, oracle/pb_oracle.c for the full-size
configurations) plus the golden vectors of tests/golden/ made from the live reference.
"""

import hashlib
import json
import os

import numpy as np
import pytest

import case_matrix
import helpers
from conftest import GOLDEN, mismatch_report

pytestmark = pytest.mark.gpu

CASES = case_matrix.all_cases()
BY_ID = {c[0]: c for c in CASES}
# Cases in which MORE than 1 % of the reference's own pixels hang on the last ulps of NumPy's libm
# (helpers.stable_pixel_mask): a property of the geometry, counted with the oracle alone by
# tests/test_oracle_golden.py::test_degenerate_case_census on the CPU -- the GPU tests may not see more.
MAX_DEGENERATE_GOLDEN = 62   # of the 585 stored reference outputs
MAX_DEGENERATE_MATRIX = 83   # of the 1701 cases


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _assert_small_case(cid, got, want, og, rots, sg, image):
    """-> (differing stable pixels [must be 0 or the 1-LSB blend class], differing pixels that
    sit on a libm-dependent boundary of the reference itself, whether the case is degenerate)."""
    from oracle import numpy_port

    if np.array_equal(got, want):
        return 0, 0, False
    diff = (got != want).reshape(got.shape[0], got.shape[1], -1).any(axis=2)
    stable = helpers.stable_pixel_mask(sg, image, numpy_port.coordinate_map(og, rots))
    degenerate = (~stable).mean() > 0.01
    hard = diff & stable
    if hard.any():
        # the only class allowed on stable pixels: 1-LSB truncation of the float64 blend of a
        # rotated double-fisheye source (SURVEY.md section 7, "blend-band rounding")
        delta = np.abs(got.astype(np.int16) - want.astype(np.int16)).reshape(diff.shape + (-1,)).max(axis=2)
        assert sg["kind"] == "double" and len(rots) > 0 and delta[hard].max() == 1 and hard.sum() <= 2, \
            (cid, int(hard.sum()), int(delta[hard].max()))
    return int(hard.sum()), int((diff & ~stable).sum()), degenerate


def test_small_matrix_against_golden_outputs(torch_cuda, golden_small):
    """585 stored reference outputs (incl. grey / RGBA layouts)."""
    meta, outputs, _ = golden_small
    n_px = n_bad = n_boundary = n_degenerate = 0
    for key in outputs.files:
        parts = key.split("__")
        cid = "__".join(parts[:3])
        _, og, rots, sg, seed = BY_ID[cid]
        channels = meta[key].get("channels", 3)
        image = case_matrix.case_image(sg, seed, channels)
        got = helpers.product_remap(og, rots, sg, image)
        want = outputs[key]
        assert got.shape == want.shape and got.dtype == np.uint8, key
        hard, boundary, degenerate = _assert_small_case(key, got, want, og, rots, sg, image)
        n_degenerate += degenerate
        if not degenerate:
            n_bad += hard + boundary
            n_px += want.shape[0] * want.shape[1]
    print(f"golden outputs: {n_bad} differing pixels of {n_px}; {n_degenerate} degenerate cases "
          f"(reference value depends on the last ulps of libm over >1% of the image) checked on their stable pixels only")
    assert n_bad / n_px <= 1e-4, (n_bad, n_px)
    # "degenerate" is a property of the reference's geometry (360-degree stereographic lenses, a
    # lat == pi row wrap over a whole row), not of this implementation: the count is pinned so that
    # a regression cannot hide behind it
    assert n_degenerate <= MAX_DEGENERATE_GOLDEN, n_degenerate


def test_small_matrix_against_numpy_oracle(torch_cuda, golden_small):
    """All 1.7k cases against oracle/numpy_port.py (itself hash-pinned to the reference)."""
    from oracle import numpy_port

    meta, _, _ = golden_small
    n_px = n_bad = n_cases_bad = n_degenerate = 0
    for cid, og, rots, sg, seed in CASES:
        image = case_matrix.case_image(sg, seed)
        want = numpy_port.remap(og, rots, sg, image)
        got = helpers.product_remap(og, rots, sg, image)
        hard, boundary, degenerate = _assert_small_case(cid, got, want, og, rots, sg, image)
        n_degenerate += degenerate
        if not degenerate:
            n_bad += hard + boundary
            n_cases_bad += (hard + boundary) > 0
            n_px += want.shape[0] * want.shape[1]
    print(f"small matrix: {n_bad} differing pixels of {n_px} in {n_cases_bad} of {len(CASES) - n_degenerate} "
          f"well-conditioned cases; {n_degenerate} degenerate cases checked on their stable pixels only")
    assert n_bad / n_px <= 1e-4, (n_bad, n_px)
    assert n_degenerate <= MAX_DEGENERATE_MATRIX, n_degenerate


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "T"])
def test_full_size_configs(torch_cuda, golden_full, name):
    """BASELINE configs at full size: CUDA vs the C oracle (run here), the reference's sha256 and
    the reference rows committed in tests/golden/full_rows_<cfg>.npz."""
    from oracle import c_port
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS[name]
    image = workloads.source_image(wl)
    assert hashlib.sha256(image.tobytes()).hexdigest() == golden_full[name]["src_sha256"]
    got = helpers.product_remap(wl["out"], wl["rotations"], wl["src"], image)
    assert list(got.shape) == golden_full[name]["shape"]

    rows = np.load(os.path.join(GOLDEN, f"full_rows_{name}.npz"))
    exact_rows, _, bad_rows = mismatch_report(got[rows["rows"]], rows["pixels"])
    assert exact_rows >= 0.9999, (name, bad_rows)

    if hashlib.sha256(got.tobytes()).hexdigest() == golden_full[name]["out_sha256"]:
        print(f"{name}: bit-identical to the reference (sha256)")
        return
    want = c_port.remap(wl["out"], wl["rotations"], wl["src"], image)
    assert hashlib.sha256(want.tobytes()).hexdigest() == golden_full[name]["out_sha256"]
    exact, max_abs, n_bad = mismatch_report(got, want)
    idx = c_port.source_index(wl["out"], wl["rotations"], wl["src"])
    n, n_flip, n_lsb, n_unexplained = helpers.attribute_mismatches(got, want, image, idx)
    print(f"{name}: exact {exact:.7f}, {n_bad} differing px: {n_flip} index flips, {n_lsb} 1-LSB, "
          f"{n_unexplained} unexplained")
    assert exact >= 0.9999, (name, exact)
    assert n_unexplained == 0, (name, n_unexplained)


def test_explicit_map_protocol(torch_cuda, golden_small):
    """get_coordinate_map -> ndarray -> rotate_coordinate_map(ndarray) -> process(ndarray):
    the materialised-map kernels agree with the fused kernel and with the reference's maps."""
    from oracle import numpy_port
    from photonbend_b200.core.rotation import Rotation

    _, _, maps = golden_small
    geoms = dict(case_matrix.output_geometries())
    rotsets = dict(case_matrix.ROTATION_SETS)
    for key in maps.files:
        oname, rname = key.split("__")
        want = maps[key]
        cmap = helpers.product_map(geoms[oname], rotsets[rname])
        got = np.asarray(cmap)
        assert got.shape == want.shape and got.dtype == np.float64
        assert np.array_equal(got[:, :, 2] != 0, want[:, :, 2] != 0), key
        valid = want[:, :, 2] == 0
        nan_ok = np.isnan(got) & np.isnan(want)
        assert np.all((np.abs(got[:, :, 0] - want[:, :, 0]) < 1e-9) | nan_ok[:, :, 0] | ~valid), key
        gx, gz = np.sin(got[:, :, 0]) * np.cos(got[:, :, 1]), np.sin(got[:, :, 0]) * np.sin(got[:, :, 1])
        wx, wz = np.sin(want[:, :, 0]) * np.cos(want[:, :, 1]), np.sin(want[:, :, 0]) * np.sin(want[:, :, 1])
        assert np.all((np.hypot(gx - wx, gz - wz) < 1e-9) | nan_ok[:, :, 0] | nan_ok[:, :, 1] | ~valid), key

    # explicit-map pipeline on a few cases, compared with the oracle image
    for cid, og, rots, sg, seed in CASES[::97]:
        image = case_matrix.case_image(sg, seed)
        want = numpy_port.remap(og, rots, sg, image)
        explicit = np.asarray(helpers.product_map(og, ()))  # materialised, unrotated
        for pyr in rots:
            explicit = Rotation(*pyr).rotate_coordinate_map(explicit)
        assert isinstance(explicit, np.ndarray)
        got = helpers.product_image(sg, image).process_coordinate_map(explicit)
        _assert_small_case(cid + " (explicit)", got, want, og, rots, sg, image)


def test_reference_side_effects_on_explicit_maps(torch_cuda):
    """rotate / panorama-process zero the invalid (lat, lon) of the map they are given."""
    from photonbend_b200.core.rotation import Rotation

    og = dict(case_matrix.output_geometries())["cam-equidistant-120"]
    cmap = np.asarray(helpers.product_map(og, ())).copy()
    invalid = cmap[:, :, 2] != 0
    assert invalid.any() and np.abs(cmap[invalid, 0]).min() > 0
    rotated = Rotation(0.1, 0.2, 0.3).rotate_coordinate_map(cmap)
    assert np.all(cmap[invalid, :2] == 0)           # input zeroed in place
    assert np.all(rotated[invalid, :2] == 0) and np.all(rotated[invalid, 2] != 0)


def test_device_batch_equals_single_frames(torch_cuda):
    """(N, H, W, C) CUDA batch: one launch, same pixels as N single-frame calls."""
    torch = torch_cuda
    from oracle import numpy_port

    sg = {"kind": "double", "height": 96, "width": 192, "lens": "equidistant",
          "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 80, "width": 160}
    frames = np.stack([case_matrix.case_image(sg, 77 + k) for k in range(5)])
    batch = torch.from_numpy(frames).cuda()
    out = helpers.product_image(sg, batch).process_coordinate_map(helpers.product_map(og, ()))
    assert out.is_cuda and tuple(out.shape) == (5, 80, 160, 3)
    out = out.cpu().numpy()
    for k in range(5):
        assert np.array_equal(out[k], numpy_port.remap(og, (), sg, frames[k])), k


def test_c_abi_direct_call(torch_cuda):
    """pb_remap_u8 called with raw device pointers, no Python host layer in between."""
    import ctypes

    torch = torch_cuda
    from oracle import numpy_port
    from photonbend_b200 import _native

    lib = _native.load()
    assert lib.pb_version() == _native.PB_ABI_VERSION
    sg = {"kind": "camera", "height": 64, "width": 64, "lens": "equidistant",
          "fov": case_matrix.rad(360), "magnitude": 31.5}
    og = {"kind": "equirect", "height": 48, "width": 96}
    image = case_matrix.case_image(sg, 5)
    d = _native.RemapDesc()
    d.out.kind, d.out.height, d.out.width = _native.KIND_EQUIRECT, 48, 96
    d.src.kind, d.src.lens, d.src.height, d.src.width = _native.KIND_CAMERA, _native.LENS_EQUIDISTANT, 64, 64
    d.src.fov = sg["fov"]
    d.src.f_distance = numpy_port.focal_distance(sg)
    d.channels, d.n_rotations = 3, 1
    mat = numpy_port.rotation_matrix(0.4, 0.5, 0.6).reshape(9)
    for e in range(9):
        d.rotations[0][e] = mat[e]
    src = torch.from_numpy(image).cuda()
    dst = torch.empty((48, 96, 3), dtype=torch.uint8, device="cuda")
    rc = lib.pb_remap_u8(ctypes.byref(d), src.data_ptr(), 64 * 64 * 3, dst.data_ptr(), 48 * 96 * 3, 1,
                         torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.pb_last_error()
    torch.cuda.synchronize()
    want = numpy_port.remap(og, [(0.4, 0.5, 0.6)], sg, image)
    assert np.array_equal(dst.cpu().numpy(), want)
    # error path: bad channel count -> code + message, no exception across the ABI
    d.channels = 7
    assert lib.pb_remap_u8(ctypes.byref(d), src.data_ptr(), 0, dst.data_ptr(), 0, 1, None) == _native.PB_ERR_UNSUPPORTED
    assert b"channels" in lib.pb_last_error()


def test_many_rotations_fall_back_to_explicit_map_kernels(torch_cuda):
    """More rotations than one launch fuses (PB_MAX_ROTATIONS) still run on the GPU."""
    from oracle import numpy_port

    sg = dict(case_matrix.source_geometries())["cam-equidistant-360"]
    og = dict(case_matrix.output_geometries())["eq"]
    rots = [(0.05 * k, -0.03 * k, 0.02 * k) for k in range(1, 20)]
    image = case_matrix.case_image(sg, 9)
    got = helpers.product_remap(og, rots, sg, image)
    want = numpy_port.remap(og, rots, sg, image)
    assert mismatch_report(got, want)[2] <= 2


def test_round_trip_property_full_size(torch_cuda):
    """Size-independent property at 8K: photo -> panorama -> photo returns every pixel of the
    inscribed circle to within one source pixel of where it started (nearest-neighbour
    resampling twice), checked on a smooth image where a one-pixel shift is a small value change."""
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["T"]
    h = wl["src"]["height"]
    yy, xx = np.mgrid[0:h, 0:h]
    smooth = np.stack([(xx * 255 // (h - 1)), (yy * 255 // (h - 1)), ((xx + yy) * 255 // (2 * h - 2))],
                      axis=2).astype(np.uint8)
    pano = helpers.product_remap(wl["out"], (), wl["src"], smooth)
    back = helpers.product_remap(wl["src"], (), wl["out"], pano)
    r = np.hypot(xx - (h - 1) / 2, yy - (h - 1) / 2)
    inside = r < h / 2 - 2
    err = np.abs(back.astype(np.int16) - smooth.astype(np.int16)).max(axis=2)
    assert err[inside].max() <= 2
    assert np.all(back[r > h / 2 + 1] == 0)  # beyond the 360-degree circle: invalid -> black


@pytest.mark.parametrize("src_kind", ["camera", "double"])
def test_tiled_fast_path_mid_size_batches(torch_cuda, src_kind):
    """The separable/TMA-staged path (16-byte aligned rows, un-rotated equirect output) on sizes
    with partial tiles, several frames per launch, against the NumPy oracle."""
    torch = torch_cuda
    from oracle import numpy_port

    if src_kind == "camera":
        sg = {"kind": "camera", "height": 400, "width": 400, "lens": "equisolid",
              "fov": case_matrix.rad(220), "magnitude": 199.5}
    else:
        sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant",
              "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 336 + 16, "width": 672 + 32}  # 11 x 11 tiles, partial edges
    frames = np.stack([case_matrix.case_image(sg, 300 + k) for k in range(3)])
    out = helpers.product_image(sg, torch.from_numpy(frames).cuda()).process_coordinate_map(
        helpers.product_map(og, ())).cpu().numpy()
    for k in range(3):
        assert np.array_equal(out[k], numpy_port.remap(og, (), sg, frames[k])), (src_kind, k)
    # one frame per launch: the persistent single-frame kernel (csrc/pb_sep1.cuh), partial edge tiles
    single = helpers.product_remap(og, (), sg, frames[1])
    assert np.array_equal(single, out[1]), src_kind
    # ... and with fewer tiles than resident CTAs, odd tile counts, a one-tile image
    for oh, ow in ((64, 32), (48, 80), (200, 1040), (65, 48)):
        og2 = {"kind": "equirect", "height": oh, "width": ow}
        assert np.array_equal(helpers.product_remap(og2, (), sg, frames[2]), numpy_port.remap(og2, (), sg, frames[2])), \
            (src_kind, oh, ow)
    # same geometry rotated: generic rays through the same tiled memory path
    rots = [(0.3, -0.7, 1.1)]
    got = helpers.product_remap(og, rots, sg, frames[0])
    want = numpy_port.remap(og, rots, sg, frames[0])
    exact, max_abs, n_bad = mismatch_report(got, want)
    # a rotated double-fisheye source may differ by the 1-LSB blend-truncation class only
    assert n_bad == 0 or (src_kind == "double" and max_abs == 1 and n_bad / (got.shape[0] * got.shape[1]) <= 1e-4), \
        (src_kind, n_bad, max_abs)
    # the same rotated geometry as a device batch: the tiled kernel with generic rays (resolved
    # once per tile, applied to every frame) must give what the single-frame direct kernel gave
    batch_out = helpers.product_image(sg, torch.from_numpy(frames[:2]).cuda()).process_coordinate_map(
        helpers.product_map(og, rots)).cpu().numpy()
    assert np.array_equal(batch_out[0], got), src_kind
    _, max_abs1, n_bad1 = mismatch_report(batch_out[1], numpy_port.remap(og, rots, sg, frames[1]))
    assert n_bad1 == 0 or (src_kind == "double" and max_abs1 == 1 and n_bad1 / (got.shape[0] * got.shape[1]) <= 1e-4), \
        (src_kind, n_bad1, max_abs1)


@pytest.mark.parametrize("fov_deg", [195, 180, 181, 210, 170, 250, 180.00000000001, 179.99999999999])
def test_double_source_batches_blend_band(torch_cuda, fov_deg, monkeypatch):
    """Batches through a double-fisheye source (csrc/pb_tiled.cuh: two launches by tile class,
    blend band through the guarded fixed-point blend) on frames chosen to sit ON the blend's
    truncation boundaries: flat frames (left == right, weights adding up to 1 -> the float64 sum is
    an integer up to its last bits), black frames, a ramp, and noise; several sensor fovs (180:
    zero-width band, division by zero in the weights; 170: negative range; within 2e-13 rad of
    180: a band so narrow that the weights grow past 2^31 and the blend leaves the int32 range of
    NumPy's uint8 cast), against the NumPy oracle."""
    torch = torch_cuda
    from oracle import numpy_port

    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": case_matrix.rad(fov_deg)}
    og = {"kind": "equirect", "height": 336 + 16, "width": 672 + 32}
    seed = round(fov_deg)
    rng = np.random.default_rng(seed)
    h, w = sg["height"], sg["width"]
    ramp = (np.arange(h * w * 3, dtype=np.int64).reshape(h, w, 3) // 7 % 256).astype(np.uint8)
    frames = np.stack([
        np.full((h, w, 3), 200, np.uint8),
        np.zeros((h, w, 3), np.uint8),
        np.full((h, w, 3), 255, np.uint8),
        ramp,
        case_matrix.case_image(sg, 500 + seed),
        (rng.integers(0, 4, (h, w, 3)) * 85).astype(np.uint8),
    ])
    want = [numpy_port.remap(og, (), sg, f) for f in frames]
    dev = torch.from_numpy(frames).cuda()
    for env in ({}, {"PB_ONE_BYTES": "4096", "PB_REST_KIB": "8"}, {"PB_CLASS_SPLIT": "0"}, {"PB_CLS2_THREADS": "256"},
                {"PB_CHUNK": "3"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        out = helpers.product_image(sg, dev).process_coordinate_map(helpers.product_map(og, ())).cpu().numpy()
        for k in range(len(frames)):
            assert np.array_equal(out[k], want[k]), (fov_deg, env, k, mismatch_report(out[k], want[k]))
        for k in env:
            monkeypatch.delenv(k)
    # one frame per call: the single-frame kernel (csrc/pb_sep1.cuh) has the same blend
    for k in (0, 3, 5):
        assert np.array_equal(helpers.product_remap(og, (), sg, frames[k]), want[k]), (fov_deg, "single", k)
    # few tiles: a class of tiles may be empty (one tile; a band that sees both lenses everywhere)
    for oh, ow in ((64, 32), (48, 80), (130, 96), (64, 704)):
        og2 = {"kind": "equirect", "height": oh, "width": ow}
        out = helpers.product_image(sg, dev[3:5]).process_coordinate_map(helpers.product_map(og2, ())).cpu().numpy()
        for k in range(2):
            assert np.array_equal(out[k], numpy_port.remap(og2, (), sg, frames[3 + k])), (fov_deg, oh, ow, k)


def _mid_size_geometries():
    """Every lens on both sides at a size that takes the tiled (TMA-staged) path."""
    rad = case_matrix.rad
    outs, srcs = [], []
    for lens, fov in (("equidistant", 360), ("equidistant", 150), ("equisolid", 180), ("equisolid", 360),
                      ("orthographic", 180), ("orthographic", 120), ("stereographic", 200),
                      ("rectilinear", 140), ("thoby", 180)):
        outs.append({"kind": "camera", "height": 200, "width": 272, "lens": lens, "fov": rad(fov),
                     "magnitude": 135.5})
        srcs.append({"kind": "camera", "height": 240, "width": 256, "lens": lens, "fov": rad(fov),
                     "magnitude": 127.5})
    for lens in ("equidistant", "equisolid", "stereographic"):
        outs.append({"kind": "double", "height": 160, "width": 320, "lens": lens, "fov": rad(195)})
        srcs.append({"kind": "double", "height": 192, "width": 384, "lens": lens, "fov": rad(190)})
    outs.append({"kind": "equirect", "height": 160, "width": 320})
    srcs.append({"kind": "equirect", "height": 192, "width": 384})
    return outs, srcs


def test_fast_path_equals_exact_chain(torch_cuda, monkeypatch):
    """csrc/pb_fast.cuh: the guarded short cut (unit-vector form, no polar round trips) must give
    the pixels of the exact chain bit for bit -- every undecided pixel falls back to it.  Checked
    on every lens pair x {no, one, two} rotations at tiled-path sizes, on the whole small matrix
    (generic kernel: rows not 16-byte aligned), and on the two rotated BASELINE configurations."""
    from photonbend_b200 import engine, workloads

    def both(og, rots, sg, image):
        monkeypatch.delenv("PB_EXACT_CHAIN", raising=False)
        engine.clear_plan_cache()
        fast = helpers.product_remap(og, rots, sg, image)
        monkeypatch.setenv("PB_EXACT_CHAIN", "1")
        engine.clear_plan_cache()
        exact = helpers.product_remap(og, rots, sg, image)
        monkeypatch.delenv("PB_EXACT_CHAIN", raising=False)
        engine.clear_plan_cache()
        return fast, exact

    outs, srcs = _mid_size_geometries()
    rotsets = ((), ((0.3, -0.2, 1.0),), ((case_matrix.rad(-90), 0.0, case_matrix.rad(195)), (0.1, 0.2, 0.3)))
    n = 0
    for a, og in enumerate(outs):
        for b, sg in enumerate(srcs):
            image = case_matrix.case_image(sg, 1000 + b)
            for rots in rotsets:
                fast, exact = both(og, rots, sg, image)
                assert np.array_equal(fast, exact), (og, rots, sg, int((fast != exact).any(axis=2).sum()))
                n += 1
    for cid, og, rots, sg, seed in CASES[::3]:
        image = case_matrix.case_image(sg, seed)
        fast, exact = both(og, rots, sg, image)
        assert np.array_equal(fast, exact), cid
        n += 1
    for name in ("cfg2", "cfg3"):
        wl = workloads.WORKLOADS[name]
        image = workloads.source_image(wl)
        fast, exact = both(wl["out"], wl["rotations"], wl["src"], image)
        assert np.array_equal(fast, exact), name
        n += 1
    print(f"short cut == exact chain on {n} cases")


def test_tiny_and_degenerate_sizes(torch_cuda):
    """One-pixel / one-row images, odd double widths, non-2:1 panoramas: the CUDA path against
    outputs of the live reference (tests/golden/make_golden_tiny.py).  On images this small many
    coordinates sit exactly on a decision boundary of the reference (a pole, a row wrap, the
    centre pixel), where its value hangs on the last ulp of NumPy's libm; those pixels are
    identified with the oracle (helpers.stable_pixel_mask) and excluded, everything else must be
    bit-exact."""
    import tiny_matrix
    from oracle import numpy_port

    with open(os.path.join(GOLDEN, "tiny_cases.json")) as fh:
        meta = json.load(fh)
    outputs = np.load(os.path.join(GOLDEN, "tiny_outputs.npz"))
    n_px = n_unstable = 0
    for cid, og, rots, sg, seed in tiny_matrix.all_cases():
        image = tiny_matrix.case_image(sg, seed)
        want = outputs[cid]
        got = helpers.product_remap(og, rots, sg, image)
        assert got.shape == want.shape and got.dtype == np.uint8, cid
        assert list(got.shape) == meta[cid]["shape"]
        if np.array_equal(got, want):
            n_px += want.shape[0] * want.shape[1]
            continue
        diff = (got != want).any(axis=2)
        stable = helpers.stable_pixel_mask(sg, image, numpy_port.coordinate_map(og, rots))
        assert not (diff & stable).any(), (cid, int((diff & stable).sum()))
        n_unstable += int(diff.sum())
        n_px += want.shape[0] * want.shape[1]
    print(f"tiny sizes: {n_px} pixels, {n_unstable} differ on libm-dependent boundaries of the reference")


def test_second_device_in_one_process(torch_cuda):
    """One process driving two GPUs (FramePipeline(device=1), tensors on cuda:1): plans, function
    attributes and tables are per device.  Skipped on a single-GPU box."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from oracle import numpy_port

    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 352, "width": 704}
    frames = np.stack([case_matrix.case_image(sg, 900 + k) for k in range(2)])
    want = [numpy_port.remap(og, (), sg, f) for f in frames]
    for dev in (0, 1, 0):
        batch = torch.from_numpy(frames).to(f"cuda:{dev}")
        out = helpers.product_image(sg, batch).process_coordinate_map(helpers.product_map(og, ()))
        assert out.device.index == dev
        single = helpers.product_image(sg, batch[1]).process_coordinate_map(helpers.product_map(og, ()))
        rotated = helpers.product_image(sg, batch[0]).process_coordinate_map(helpers.product_map(og, [(0.3, -0.7, 1.1)]))
        assert np.array_equal(out.cpu().numpy()[0], want[0]) and np.array_equal(out.cpu().numpy()[1], want[1]), dev
        assert np.array_equal(single.cpu().numpy(), want[1]), dev
        # a rotated double-fisheye source: only the 1-LSB blend-truncation class may differ
        _, max_abs, n_bad = mismatch_report(rotated.cpu().numpy(), numpy_port.remap(og, [(0.3, -0.7, 1.1)], sg, frames[0]))
        assert n_bad == 0 or (max_abs == 1 and n_bad <= 25), (dev, n_bad, max_abs)


@pytest.mark.parametrize("rots", [(), ((0.3, -0.7, 1.1),)], ids=["separable", "rotated"])
def test_row_bands_equal_the_whole_frame(torch_cuda, rots):
    """pb_plan_remap_rows_u8 / batch.remap_row_band: a frame cut into output-row bands (tile-aligned
    ones from shard_rows, and odd ones) gives exactly the rows of the whole-frame remap."""
    torch = torch_cuda
    from photonbend_b200.batch import remap_row_band, shard_rows

    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 420, "width": 704}
    frame = torch.from_numpy(case_matrix.case_image(sg, 77)).cuda()
    source = helpers.product_image(sg, frame)
    cmap = helpers.product_map(og, rots)
    whole = source.process_coordinate_map(cmap).cpu().numpy()
    for world in (1, 2, 3, 8):
        bands = [remap_row_band(source, cmap, frame, shard_rows(og["height"], r, world)) for r in range(world)]
        got = torch.cat(bands, dim=0).cpu().numpy()
        assert np.array_equal(got, whole), (rots, world)
    for rows in (range(0, 1), range(5, 133), range(64, 65), range(419, 420), range(100, 100)):
        band = remap_row_band(source, cmap, frame, rows).cpu().numpy()
        assert np.array_equal(band, whole[rows.start:rows.stop]), (rots, rows)


def _cfg5_frames(n):
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["cfg5"]
    with open(os.path.join(GOLDEN, "cfg5_frames.json")) as fh:
        golden = json.load(fh)["frames"]
    frames = []
    for k in range(n):
        image = workloads.source_image(wl, frame=k)
        assert hashlib.sha256(image.tobytes()).hexdigest() == golden[k]["src_sha256"], k
        frames.append(image)
    return wl, golden, frames


@pytest.mark.parametrize("concurrent", ["1", "0"], ids=["two-grids-concurrent", "two-grids-in-sequence"])
def test_cfg5_full_size_batch(torch_cuda, monkeypatch, concurrent):
    """BASELINE config 5 as bench.py runs it: distinct full-size (3840x7680) double-fisheye frames
    (seeds 1234 + k) through ONE remap_batch call -- the class-split batched kernel, census-picked
    stage sizes, both grids (on two streams, and in sequence with PB_CONCURRENT=0) -- every frame's
    sha256 against the live reference's (tests/golden/cfg5_frames.json, made by
    tests/golden/make_golden_cfg5.py from the unmodified reference, projection.py:408-462)."""
    torch = torch_cuda
    from photonbend_b200 import engine
    from photonbend_b200.batch import remap_batch

    monkeypatch.setenv("PB_CONCURRENT", concurrent)
    engine.clear_plan_cache()
    n = 6
    wl, golden, frames = _cfg5_frames(n)
    batch = torch.from_numpy(np.stack(frames)).cuda()
    source = helpers.product_image(wl["src"], batch)
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    out = remap_batch(source, cmap, batch)
    out2 = remap_batch(source, cmap, batch, torch.empty_like(out))  # a second launch into another buffer
    torch.cuda.synchronize()
    assert torch.equal(out, out2)
    out = out.cpu().numpy()
    for k in range(n):
        got = hashlib.sha256(out[k].tobytes()).hexdigest()
        if got != golden[k]["out_sha256"]:
            from oracle import c_port

            want = c_port.remap(wl["out"], wl["rotations"], wl["src"], frames[k])
            assert hashlib.sha256(want.tobytes()).hexdigest() == golden[k]["out_sha256"], ("oracle vs reference", k)
            raise AssertionError((concurrent, k, mismatch_report(out[k], want)))
    engine.clear_plan_cache()


@pytest.mark.parametrize("batch", [1, 3], ids=["launch-per-frame", "three-frames-per-launch"])
def test_frame_pipeline_full_size(torch_cuda, batch):
    """batch.FramePipeline (the API bench.py's e2e figure is quoted through): depth 3, eight pinned
    host frames of config 5 in, eight pinned host frames out, per-frame sha256 against the live
    reference.  Three streams share one plan (tensor-map cache, side-stream lanes); with batch=3
    the last launch is a partly filled batch (8 = 3 + 3 + 2)."""
    torch = torch_cuda
    from photonbend_b200.batch import FramePipeline

    n = 8
    wl, golden, frames = _cfg5_frames(n)
    host_in = []
    for f in frames:
        t = torch.empty(f.shape, dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = f
        host_in.append(t)
    oh, ow, _ = workloads_shape(wl)
    host_out = [torch.zeros((oh, ow, 3), dtype=torch.uint8, pin_memory=True) for _ in range(n)]
    source = helpers.product_image(wl["src"], frames[0])
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    pipe = FramePipeline(source, cmap, depth=3, batch=batch)
    for rounds in range(2):  # the second round reuses every device buffer and cached tensor map
        pipe.run(host_in, host_out)
        for k in range(n):
            assert hashlib.sha256(host_out[k].numpy().tobytes()).hexdigest() == golden[k]["out_sha256"], (batch, rounds, k)
            host_out[k].zero_()
    assert pipe.kernel_launches == 2 * (n if batch == 1 else 3)


def workloads_shape(wl):
    from photonbend_b200 import workloads

    return workloads.output_shape(wl["out"])


def test_plan_less_abi_wide_short_footprints(torch_cuda):
    """pb_remap_u8 WITHOUT a plan (the documented drop-in entry point) on an un-rotated equirect
    output whose tiles have wide, short source footprints (21..31 sixteen-byte units): every box
    width needs its tensor map although no census ran (ADVICE round 1: the single-frame kernel
    indexed maps that were never encoded).  Several tile rows, one frame and a batch."""
    import ctypes

    torch = torch_cuda
    from oracle import numpy_port
    from photonbend_b200 import _native

    lib = _native.load()
    for (sh, sw, oh, ow, lens, fov) in ((2048, 2048, 2048, 1024, "equidistant", 360), (1024, 1024, 640, 256, "equisolid", 300),
                                        (1536, 1536, 1024, 512, "stereographic", 200)):
        sg = {"kind": "camera", "height": sh, "width": sw, "lens": lens, "fov": case_matrix.rad(fov),
              "magnitude": sw / 2 - 0.5}
        og = {"kind": "equirect", "height": oh, "width": ow}
        d = _native.RemapDesc()
        d.out.kind, d.out.height, d.out.width = _native.KIND_EQUIRECT, oh, ow
        d.src.kind, d.src.height, d.src.width = _native.KIND_CAMERA, sh, sw
        d.src.lens = numpy_port.LENS_NAMES.index(lens)
        d.src.fov = sg["fov"]
        d.src.f_distance = numpy_port.focal_distance(sg)
        d.channels, d.n_rotations = 3, 0
        images = np.stack([case_matrix.case_image(sg, 40 + k) for k in range(2)])
        src = torch.from_numpy(images).cuda()
        for n_frames in (1, 2):
            dst = torch.zeros((n_frames, oh, ow, 3), dtype=torch.uint8, device="cuda")
            rc = lib.pb_remap_u8(ctypes.byref(d), src.data_ptr(), sh * sw * 3, dst.data_ptr(), oh * ow * 3, n_frames,
                                 torch.cuda.current_stream().cuda_stream)
            assert rc == 0, lib.pb_last_error()
            torch.cuda.synchronize()
            got = dst.cpu().numpy()
            for k in range(n_frames):
                assert np.array_equal(got[k], numpy_port.remap(og, (), sg, images[k])), (lens, n_frames, k)


def test_plan_shared_by_host_threads(torch_cuda):
    """One geometry remapped from four host threads at once, each on its own CUDA stream (ctypes
    releases the GIL inside the call): launches through one pb_plan are serialised inside the
    library (tensor-map caches, side-stream lanes), results are those of the oracle."""
    import threading

    torch = torch_cuda
    from oracle import numpy_port

    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 352, "width": 704}
    images = [case_matrix.case_image(sg, 700 + k) for k in range(4)]
    want = [numpy_port.remap(og, (), sg, im) for im in images]
    cmap = helpers.product_map(og, ())
    helpers.product_image(sg, torch.from_numpy(images[0]).cuda()).process_coordinate_map(cmap)  # plan exists
    errors = []

    def worker(k):
        try:
            stream = torch.cuda.Stream()
            with torch.cuda.stream(stream):
                dev = torch.from_numpy(images[k]).cuda()
                for _ in range(25):
                    out = helpers.product_image(sg, dev).process_coordinate_map(cmap)
                stream.synchronize()
                if not np.array_equal(out.cpu().numpy(), want[k]):
                    errors.append(k)
        except Exception as exc:  # noqa: BLE001
            errors.append(repr(exc))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


def fp32_tier_stats(og, rots, sg):
    """pb_debug_fast32_stats for a geometry: dict(max_ratio_x, max_ratio_y, pixels, undecided, wrong, status_mismatch)."""
    import ctypes

    from photonbend_b200 import _native, engine

    cmap = helpers.product_map(og, rots)
    src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
    desc = engine._remap_desc(cmap.rays, src._source_geometry(), 3)
    stats = (ctypes.c_double * 6)()
    _native.check(_native.load().pb_debug_fast32_stats(ctypes.byref(desc), stats, None))
    keys = ("max_ratio_x", "max_ratio_y", "pixels", "undecided", "wrong", "status_mismatch")
    return dict(zip(keys, [float(v) for v in stats]))


FP32_TIER_K = 16.0  # csrc/pb_remap.cu kFast32K


def test_fp32_tier_error_bound(torch_cuda):
    """csrc/pb_fast32.cuh: the FP32-first tier accepts a pixel only if its float coordinate is
    further than E = K * 2^-24 * shape from every integer.  Over every pixel of every lens pair x
    {no, one, two} rotations at mid size, a third of the small matrix and the two rotated BASELINE
    configurations at full size: (1) the float evaluation never strays from the float64 evaluation of
    the same formulas by more than HALF the bound (max ratio <= K / 2), (2) no pixel tier 1 decides
    differs from what the float64 tiers give, (3) float and double agree on every fov / no-pixel
    decision tier 1 takes."""
    from photonbend_b200 import workloads

    outs, srcs = _mid_size_geometries()
    rotsets = ((), ((0.3, -0.2, 1.0),), ((case_matrix.rad(-90), 0.0, case_matrix.rad(195)), (0.1, 0.2, 0.3)))
    worst, n_px, n_und, n_cases = 0.0, 0.0, 0.0, 0
    geoms = [(og, rots, sg) for og in outs for sg in srcs for rots in rotsets]
    geoms += [(og, rots, sg) for _, og, rots, sg, _ in CASES[::3]]
    geoms += [(workloads.WORKLOADS[n]["out"], workloads.WORKLOADS[n]["rotations"], workloads.WORKLOADS[n]["src"])
              for n in ("cfg2", "cfg3", "cfg1", "cfg4")]
    for og, rots, sg in geoms:
        try:
            st = fp32_tier_stats(og, rots, sg)
        except ValueError:
            continue  # a geometry the reference refuses at construction (rectilinear fov)
        assert st["wrong"] == 0 and st["status_mismatch"] == 0, (og, rots, sg, st)
        worst = max(worst, st["max_ratio_x"], st["max_ratio_y"])
        assert max(st["max_ratio_x"], st["max_ratio_y"]) <= FP32_TIER_K / 2, (og, rots, sg, st)
        n_px += st["pixels"]
        n_und += st["undecided"]
        n_cases += 1
    print(f"FP32 tier: {n_cases} geometries, {n_px:.0f} pixels, largest |float - double| / (2^-24 shape) = {worst:.2f} "
          f"(bound K = {FP32_TIER_K}), {n_und / n_px:.4f} of the pixels left to the float64 tiers")


def test_plan_calibrates_the_fp32_bound(torch_cuda, monkeypatch):
    """pb_plan_create measures |float - double| / (2^-24 shape) over the plan's own pixels and bounds
    tier 1 with K = max(1.5, 1.25 ratio + 0.25) instead of the K = 16 that holds for every geometry.
    For the two rotated BASELINE configurations and three mid-size lens pairs: the plan reports the
    ratio pb_debug_fast32_stats measures, its K is the formula's, and with THAT K (PB_FP32_K, read
    by the diagnostics too) tier 1 still decides no pixel differently from the float64 tiers while
    leaving fewer undecided.  Separable plans (tables) do not calibrate."""
    import ctypes

    import torch

    from photonbend_b200 import _native, engine, workloads

    lib = _native.load()
    outs, srcs = _mid_size_geometries()
    geoms = [(workloads.WORKLOADS[n]["out"], workloads.WORKLOADS[n]["rotations"], workloads.WORKLOADS[n]["src"])
             for n in ("cfg2", "cfg3")]
    geoms += [(outs[k % len(outs)], ((0.3, -0.2, 1.0),), srcs[(2 * k + 1) % len(srcs)]) for k in range(3)]
    for og, rots, sg in geoms:
        monkeypatch.delenv("PB_FP32_K", raising=False)
        try:
            base = fp32_tier_stats(og, rots, sg)
        except ValueError:
            continue
        cmap = helpers.product_map(og, rots)
        src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
        desc = engine._remap_desc(cmap.rays, src._source_geometry(), 3)
        plan = engine._plans.get(lib, desc, torch.cuda.current_device(), torch)
        got = (ctypes.c_double * 2)()
        _native.check(lib.pb_debug_plan_fast32(plan, got))
        k_plan, ratio = float(got[0]), float(got[1])
        if sg["kind"] == "double" and not rots:
            continue
        want_ratio = max(base["max_ratio_x"], base["max_ratio_y"])
        assert abs(ratio - want_ratio) <= 1e-3 * max(1.0, want_ratio), (og, sg, ratio, want_ratio)
        assert k_plan == pytest.approx(max(1.5, 1.25 * ratio + 0.25), rel=1e-6) and k_plan <= 16.0, (og, sg, k_plan)
        monkeypatch.setenv("PB_FP32_K", repr(k_plan))
        tight = fp32_tier_stats(og, rots, sg)
        assert tight["wrong"] == 0 and tight["status_mismatch"] == 0, (og, sg, tight)
        assert tight["undecided"] <= base["undecided"], (og, sg, tight["undecided"], base["undecided"])
        print(f"{og['kind']} <- {sg['kind']}: ratio {ratio:.2f}, K {k_plan:.2f}, undecided {base['undecided'] / base['pixels']:.4f} "
              f"-> {tight['undecided'] / tight['pixels']:.4f}")
    monkeypatch.delenv("PB_FP32_K", raising=False)
    # an un-rotated panorama output through a camera source resolves through tables: nothing to calibrate
    og, sg = {"kind": "equirect", "height": 128, "width": 256}, srcs[0]
    if sg["kind"] == "camera":
        src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
        desc = engine._remap_desc(helpers.product_map(og, ()).rays, src._source_geometry(), 3)
        plan = engine._plans.get(lib, desc, torch.cuda.current_device(), torch)
        got = (ctypes.c_double * 2)()
        _native.check(lib.pb_debug_plan_fast32(plan, got))
        assert float(got[1]) == -1.0


def test_map_projection_on_device(torch_cuda, golden_small):
    """core.map_projection (pb_map_projection_u8, reference projection.py:550-599): bit-identical to
    the live reference's outputs on the reference's own maps (ndarray argument: uploaded, invalid
    entries zeroed in place like the reference does), and within rounding of them on the map the
    device materialises itself (CUDA's libm differs from NumPy's in the last ulp, which can move a
    value across a .5 rounding boundary)."""
    from photonbend_b200.core import map_projection

    _, _, maps = golden_small
    golden = np.load(os.path.join(GOLDEN, "map_projection.npz"))
    geoms = dict(case_matrix.output_geometries())
    rotsets = dict(case_matrix.ROTATION_SETS)
    n_px = n_off = 0
    for key in golden.files:
        cmap = maps[key].copy()
        got = map_projection(cmap)
        assert got.dtype == np.uint8 and np.array_equal(got, golden[key]), key
        assert np.all(cmap[cmap[:, :, 2] != 0, :2] == 0), key
        oname, rname = key.split("__")
        if "stereographic-360" in oname:
            continue  # infinite image radius: the largest latitude (the stretch of the red channel) hangs on the last ulp of libm
        lazy = map_projection(helpers.product_map(geoms[oname], rotsets[rname]))
        diff = np.abs(lazy.astype(np.int16) - golden[key].astype(np.int16))
        diff = np.minimum(diff, 256 - diff)  # the green channel wraps (negative longitudes)
        # the +-pi seam: a longitude of pi - 1e-16 shows as 127, one of -pi + 1e-16 as 129
        seam = np.isin(lazy[:, :, 1], (127, 128, 129)) & np.isin(golden[key][:, :, 1], (127, 128, 129))
        diff[:, :, 1][seam] = 0
        assert diff.max() <= 1, (key, int(diff.max()), int((diff > 1).sum()))
        n_px += diff[:, :, 0].size
        n_off += int((diff > 0).any(axis=2).sum())
    assert n_off <= 2e-3 * n_px, (n_off, n_px)
    with pytest.raises(ValueError):
        map_projection(np.ones((4, 4, 3)))  # no valid pixel: numpy.min of an empty selection


def test_user_defined_lens_through_tables(torch_cuda):
    """A Lens built from user callables (reference lens.py:48-64) runs on the GPU through a table of
    samples (PB_LENS_TABLE, linear interpolation; include/pb_remap.h).  With callables that compute
    what a built-in model computes, the pixels are those of the built-in model except where the
    interpolation error (~1e-7 px) moves a coordinate across an integer: at most a handful of
    pixels, each the neighbouring source pixel.  Fused path (both roles, rotated and not, one frame
    and a batch) and the explicit-map path."""
    torch = torch_cuda
    from photonbend_b200.core.lens import Lens, equisolid, stereographic
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, PanoramaImage
    from photonbend_b200.core.rotation import Rotation

    pairs = [
        (equisolid(), Lens(lambda t: 2 * np.sin(t / 2), lambda r: 2 * np.arcsin(r / 2))),
        (stereographic(), Lens(lambda t: 2 * np.tan(t / 2), lambda r: 2 * np.arctan(r / 2))),
    ]
    rng = np.random.default_rng(11)
    photo = rng.integers(0, 256, (240, 256, 3), dtype=np.uint8)
    pano = rng.integers(0, 256, (192, 384, 3), dtype=np.uint8)
    dbl = rng.integers(0, 256, (192, 384, 3), dtype=np.uint8)
    n_px = n_bad = 0
    for builtin, custom in pairs:
        for rot in (None, (0.3, -0.2, 1.0)):
            results = []
            for lens in (builtin, custom):
                outs = []
                # custom lens as the SOURCE: photo -> panorama, double -> panorama
                cmap = PanoramaImage(np.zeros((160, 320, 3), np.uint8)).get_coordinate_map()
                if rot:
                    cmap = Rotation(*rot).rotate_coordinate_map(cmap)
                outs.append(CameraImage(photo, case_matrix.rad(200), lens, magnitude=127.5).process_coordinate_map(cmap))
                outs.append(DoubleCameraImage(dbl, case_matrix.rad(195), lens).process_coordinate_map(cmap))
                # custom lens as the OUTPUT: panorama -> photo
                cmap = CameraImage(np.zeros((200, 272, 3), np.uint8), case_matrix.rad(150), lens, magnitude=135.5).get_coordinate_map()
                if rot:
                    cmap = Rotation(*rot).rotate_coordinate_map(cmap)
                outs.append(PanoramaImage(pano).process_coordinate_map(cmap))
                # explicit map: materialised with the custom reverse function, gathered with the custom forward
                explicit = np.asarray(cmap).copy()
                outs.append(CameraImage(photo, case_matrix.rad(200), lens, magnitude=127.5).process_coordinate_map(explicit))
                # a device batch through the custom source lens
                batch = torch.from_numpy(np.stack([photo, photo[::-1].copy()])).cuda()
                cmap = PanoramaImage(np.zeros((160, 320, 3), np.uint8)).get_coordinate_map()
                outs.append(CameraImage(batch, case_matrix.rad(200), lens, magnitude=127.5).process_coordinate_map(cmap).cpu().numpy())
                results.append(outs)
            for a, b in zip(*results):
                assert a.shape == b.shape
                diff = (a != b).any(axis=-1)
                n_px += diff.size
                n_bad += int(diff.sum())
    print(f"user-defined lens tables: {n_bad} of {n_px} pixels differ from the built-in model")
    assert n_bad <= max(4, 2e-5 * n_px), (n_bad, n_px)


def test_non_orthonormal_matrices_take_the_exact_chain(torch_cuda, monkeypatch):
    """The raw ABI takes any 9 doubles as a rotation.  The short cuts carry the ray as a unit vector
    through ONE composed matrix, which equals the reference's per-rotation acos / atan2 round trip
    only for orthonormal matrices: anything else must switch them off (derive_fast) and give what
    the exact chain gives (ADVICE round 1)."""
    import ctypes

    torch = torch_cuda
    from oracle import numpy_port
    from photonbend_b200 import _native, engine

    lib = _native.load()
    sg = {"kind": "camera", "height": 256, "width": 256, "lens": "equidistant", "fov": case_matrix.rad(360), "magnitude": 127.5}
    image = case_matrix.case_image(sg, 21)
    src = torch.from_numpy(image).cuda()
    d = _native.RemapDesc()
    d.out.kind, d.out.height, d.out.width = _native.KIND_EQUIRECT, 192, 384
    d.src.kind, d.src.lens, d.src.height, d.src.width = _native.KIND_CAMERA, _native.LENS_EQUIDISTANT, 256, 256
    d.src.fov, d.src.f_distance = sg["fov"], numpy_port.focal_distance(sg)
    d.channels, d.n_rotations = 3, 2
    rot = numpy_port.rotation_matrix(0.4, 0.5, 0.6)
    shear = rot @ np.array([[1.0, 0.2, 0.0], [0.0, 0.9, 0.0], [0.0, 0.0, 1.0]])  # scaled and sheared
    for k, m in enumerate((shear, rot)):
        for e in range(9):
            d.rotations[k][e] = m.reshape(9)[e]

    def run():
        dst = torch.zeros((192, 384, 3), dtype=torch.uint8, device="cuda")
        rc = lib.pb_remap_u8(ctypes.byref(d), src.data_ptr(), 0, dst.data_ptr(), 0, 1, torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.pb_last_error()
        torch.cuda.synchronize()
        return dst.cpu().numpy()

    got = run()
    monkeypatch.setenv("PB_EXACT_CHAIN", "1")
    exact = run()
    monkeypatch.delenv("PB_EXACT_CHAIN")
    assert np.array_equal(got, exact)
    stats = (ctypes.c_double * 6)()
    assert lib.pb_debug_fast32_stats(ctypes.byref(d), stats, None) == 0
    assert stats[3] == stats[2], "tier 1 must leave every pixel of a non-orthonormal remap undecided"
    engine.clear_plan_cache()


def _random_geometry(rng, role):
    """A random mid-size geometry (several tiles, odd edges) away from the degenerate corners the
    census of tests/test_oracle_golden.py counts (360-degree stereographic, rectilinear >= 175)."""
    kind = rng.choice(["equirect", "camera", "double"])
    if kind == "equirect":
        h = int(rng.integers(48, 260))
        return {"kind": "equirect", "height": h, "width": 2 * h + int(rng.choice([0, 0, 1, 6, 16]))}
    lens = str(rng.choice(["equidistant", "equisolid", "orthographic", "stereographic", "rectilinear", "thoby"]))
    hi = {"orthographic": 180, "stereographic": 280, "rectilinear": 165, "thoby": 220}.get(lens, 360)
    lo = 60 if lens == "rectilinear" else 100
    if kind == "double":
        if lens in ("rectilinear", "orthographic"):
            lens = "equidistant"
            lo, hi = 170, 250
        else:
            lo, hi = 170, min(hi, 250)
        h = int(rng.integers(60, 280))
        return {"kind": "double", "height": h, "width": 2 * h + int(rng.choice([0, 0, 1, 8])), "lens": lens,
                "fov": case_matrix.rad(float(rng.uniform(lo, hi)))}
    h, w = int(rng.integers(60, 420)), int(rng.integers(60, 420))
    if rng.random() < 0.5:
        w = h
    mag = None if rng.random() < 0.4 else float(rng.uniform(0.4, 0.75) * min(h, w))
    return {"kind": "camera", "height": h, "width": w, "lens": lens, "fov": case_matrix.rad(float(rng.uniform(lo, hi))),
            "magnitude": mag}


@pytest.mark.parametrize("fuzz_seed", [20261018, 7, 990])
def test_random_mid_size_geometries(torch_cuda, fuzz_seed):
    """Seeded fuzz (three seeds): 60 random (output, rotations, source) triples at sizes of several tiles -- every
    kernel family gets some (separable batches and single frames when un-rotated, the FP32-first
    rotated kernel, two-lens tiles, explicit maps for > 8 rotations never) -- against
    oracle/numpy_port.py (bit-identical to the reference).  Same acceptance as the small matrix."""
    torch = torch_cuda
    from oracle import c_port, numpy_port

    rng = np.random.default_rng(fuzz_seed)
    n_px = n_bad = n_degenerate = n_lsb = 0
    for case in range(60):
        og, sg = _random_geometry(rng, "out"), _random_geometry(rng, "src")
        n_rot = int(rng.choice([0, 0, 1, 2]))
        rots = tuple(tuple(float(v) for v in rng.uniform(-3.2, 3.2, 3)) for _ in range(n_rot))
        n_frames = int(rng.choice([1, 1, 3]))
        frames = np.stack([case_matrix.case_image(sg, 7000 + 10 * case + k) for k in range(n_frames)])
        src = helpers.product_image(sg, torch.from_numpy(frames if n_frames > 1 else frames[0]).cuda())
        got = src.process_coordinate_map(helpers.product_map(og, rots)).cpu().numpy()
        got = got if n_frames > 1 else got[None]
        for k in range(n_frames):
            want = numpy_port.remap(og, rots, sg, frames[k])
            cid = f"fuzz{case}.{k} {og} {rots} {sg}"
            assert got[k].shape == want.shape, cid
            if np.array_equal(got[k], want):
                n_px += want.shape[0] * want.shape[1]
                continue
            diff = (got[k] != want).any(axis=2)
            stable = helpers.stable_pixel_mask(sg, frames[k], numpy_port.coordinate_map(og, rots))
            if (~stable).mean() > 0.01:
                n_degenerate += 1
                assert not (diff & stable).any() or sg["kind"] == "double", cid
                continue
            hard = diff & stable
            if hard.any():
                # only the 1-LSB class of a double-fisheye source: a float64 blend v0 w0 + v1 w1 whose exact
                # value is an integer (v0 == v1 in some channel, w0 + w1 == 1) truncates to v or v - 1 on the
                # last ulp of the weights, i.e. of libm's sin / cos / atan2 (SURVEY.md section 7)
                # -- noise images make it as frequent as it gets (3 / 256 of the blended pixels are exposed)
                delta = np.abs(got[k].astype(np.int16) - want.astype(np.int16)).max(axis=2)
                assert sg["kind"] == "double" and delta[hard].max() == 1 and hard.mean() <= 2e-4, (cid, int(hard.sum()))
                idx = c_port.source_index(og, rots, sg)
                assert (idx[hard] >= 0).all(), cid  # every one of them blends two source pixels
                n_lsb += int(hard.sum())
            n_bad += int(diff.sum())
            n_px += want.shape[0] * want.shape[1]
    print(f"fuzz: {n_bad} differing pixels of {n_px} ({n_lsb} of the 1-LSB blend class); {n_degenerate} degenerate draws")
    assert n_bad / n_px <= 1e-4, (n_bad, n_px)
    assert n_degenerate <= 6, n_degenerate
