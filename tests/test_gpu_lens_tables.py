"""User-defined lenses (PB_LENS_TABLE) on every kernel route, bit for bit against the table oracle
(tests/table_oracle.py): numpy_port with each per-pixel lens evaluation replaced by the interpolation of
the table the product built, which the kernels must reproduce exactly (lens_table_at, -fmad=false).

The lenses are not the built-in models: a Kannala-Brandt polynomial with a Newton inverse, a
non-monotone wavy lens, a lens that is NaN beyond 80 degrees, and a forward / reverse pair that are not
inverses of each other (a route that reads the other side's table gives other pixels).  Tables of 2, 3,
17, 1025 and 65537 samples (core.projection.lens_table patched to that length): on coarse tables every
interpolation step moves pixels.  Every product call reads the launch census, so each route this file
claims is the one that ran.  Acceptance: helpers.Oracle (bit-exact on the pixels whose value does not
hang on the last ulps of libm; a double-fisheye source may differ by the 1-LSB blend class only)."""

import ctypes
import functools
import math

import numpy as np
import pytest

import helpers
import table_oracle
import typed_oracle

pytestmark = pytest.mark.gpu

rad = np.deg2rad
OUT_H, OUT_W = 170, 336  # partial tiles on the right and bottom edges
SAMPLES = (2, 3, 17, 1025, 65537)
ROT = ((0.3, -0.2, 1.0),)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(autouse=True)
def _table_oracle():
    with table_oracle.patched():
        yield


# ------------------------------------------------------------------------------------ lenses

K1, K2 = 0.08, 0.01


def _kb(t):
    return t * (1 + K1 * t**2 + K2 * t**4)


def _kb_inverse(r):
    r = np.asarray(r, dtype=np.float64)
    t = r.copy()
    for _ in range(30):  # Newton on theta (1 + k1 theta^2 + k2 theta^4) = r; monotone for k1, k2 > 0
        t = t - (_kb(t) - r) / (1 + 3 * K1 * t**2 + 5 * K2 * t**4)
    return t


def _nan80(t):
    t = np.asarray(t, dtype=np.float64)
    return np.where(t > rad(80), np.nan, 2 * np.sin(t / 2))


def _nan80_inverse(r):
    t = 2 * np.arcsin(np.asarray(r, dtype=np.float64) / 2)
    return np.where(t > rad(80), np.nan, t)


# (forward, reverse, camera fov in degrees, double-fisheye sensor fov or None)
LENSES = {
    "kb": (_kb, _kb_inverse, 200, 195),
    "wavy": (lambda t: t + 0.2 * np.sin(6 * t), lambda r: r - 0.2 * np.sin(6 * r), 190, 190),  # d/dt < 0 in places
    "nan80": (_nan80, _nan80_inverse, 150, None),
    "mismatched": (lambda t: 2 * np.sin(t / 2), lambda r: 1.1 * r, 180, 200),  # not inverses of each other
}


def _lens(name):
    from photonbend_b200.core.lens import Lens

    fwd, rev = LENSES[name][:2]
    return Lens(fwd, rev)


def _with_samples(n, fn):
    """fn() with core.projection.lens_table sampling n points (LENS_TABLE_SAMPLES is bound as a default)"""
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core import projection

    saved = projection.lens_table
    projection.lens_table = functools.partial(pb_lens.lens_table, samples=n)
    try:
        return fn()
    finally:
        projection.lens_table = saved


def _image(kind, lens, n, role, array, keep_dtype=False):
    """A product image of ``kind`` whose table for ``role`` has n samples (lens None: built-in)"""
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, PanoramaImage

    if kind == "equirect":
        return PanoramaImage(array)
    user = _lens(lens) if lens else pb_lens.equisolid()
    if kind == "camera":
        fov = LENSES[lens][2] if lens else 180
        image = CameraImage(array, rad(fov), user, magnitude=150.5 if role == "output" else 119.5)
    else:
        fov = (LENSES[lens][3] or 195) if lens else 190
        image = DoubleCameraImage(array, rad(fov), user, keep_dtype=keep_dtype)
    if lens:
        _with_samples(n, image._output_geometry if role == "output" else image._source_geometry)
    return image


def _frames(shape, n, seed, dtype=np.uint8):
    """noise, flat and ramp frames"""
    rng = np.random.default_rng(seed)
    h, w, c = shape
    ramp = np.arange(h * w * c, dtype=np.int64).reshape(h, w, c) // 5
    out = []
    for k in range(n):
        if k % 3 == 0:
            out.append(rng.integers(0, 256, shape, dtype=np.uint8))
        elif k % 3 == 1:
            out.append(np.full(shape, (200 + 37 * k) % 256, np.uint8))
        else:
            out.append(((ramp + 13 * k) % 256).astype(np.uint8))
    frames = np.stack(out)
    if dtype != np.uint8:
        frames = (frames.astype(np.float64) * 3.25 - 100).astype(dtype)
    return frames


class Case:
    """One remap: output image (its rays), rotations, source image; the oracle's geometries"""

    def __init__(self, okind, olens, rots, skind, slens, n_out=17, n_src=1025, channels=3, sshape=None,
                 keep_dtype=False):
        sshape = sshape or {"camera": (240, 256), "double": (192, 384), "equirect": (192, 384)}[skind]
        self.out_img = _image(okind, olens, n_out, "output", np.zeros((OUT_H, OUT_W, 3), np.uint8))
        self.src_shape = sshape + (channels,)
        self.src_img = _image(skind, slens, n_src, "source", np.zeros(self.src_shape, np.uint8), keep_dtype)
        self.rots = rots
        self.og, self.sg = table_oracle.geom_of(self.out_img), table_oracle.geom_of(self.src_img)
        self.cid = f"{okind}-{olens}/{n_out}{list(rots)}<-{skind}-{slens}/{n_src}"

    def cmap(self):
        from photonbend_b200.core.rotation import Rotation

        cmap = self.out_img.get_coordinate_map()
        for pyr in self.rots:
            cmap = Rotation(*pyr).rotate_coordinate_map(cmap)
        return cmap

    def source(self, array):
        image = self.src_img
        image.image = array
        return image

    def run(self, array):
        """-> (numpy output, census) of process_coordinate_map on ``array`` (a CUDA tensor)"""
        cmap = self.cmap()
        out, ran = helpers.remap_launches(lambda: self.source(array).process_coordinate_map(cmap))
        return out.cpu().numpy(), ran

    def oracle(self):
        return helpers.Oracle(self.og, self.rots, self.sg)

    def check(self, got, frames, what=""):
        oracle = self.oracle()
        for k in range(len(frames)):
            oracle.check(_bytes(got[k]), _bytes(frames[k]), (self.cid, what, k))
        oracle.assert_lsb_share()


def _bytes(a):
    """(H, W, C) of any dtype -> (H, W, C * itemsize) uint8: the oracle picks the same pixels"""
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(a.shape[0], a.shape[1], -1)


def _lens_cycle(k, double=False):
    names = [n for n in LENSES if not double or LENSES[n][3]]
    return names[k % len(names)]


# ------------------------------------------------------------------------------------ fused routes

# (route, output kind, rotated, source kind, sides, frames, 1-byte source offset, expected families)
ROUTES = [
    ("sep1-camera", "equirect", False, "camera", ("source",), 1, False, {"sep1"}),
    ("sep1-double", "equirect", False, "double", ("source",), 1, False, {"sep1"}),
    ("direct", "equirect", True, "camera", ("source",), 1, False, {"direct"}),
    ("direct", "camera", True, "equirect", ("output",), 1, False, {"direct"}),
    ("direct", "camera", False, "camera", ("both",), 1, False, {"direct"}),
    ("direct", "double", True, "double", ("output", "both"), 1, False, {"direct"}),
    ("generic", "equirect", False, "camera", ("source",), 1, True, {"generic"}),
    ("generic", "camera", True, "camera", ("output", "both"), 9, True, {"generic"}),
    ("tiled_sep", "equirect", False, "camera", ("source",), 9, False, {"tiled_sep"}),
    ("boxes", "equirect", False, "double", ("source",), 9, False, {"boxes1", "boxes2"}),
    ("tiled", "equirect", True, "double", ("source",), 9, False, {"tiled"}),
    ("tiled", "camera", False, "equirect", ("output",), 9, False, {"tiled"}),
    ("tiled", "double", True, "camera", ("both",), 9, False, {"tiled"}),
    ("tiled", "camera", False, "double", ("both",), 9, False, {"tiled"}),
]


def _route_cases():
    cases = []
    k = 0
    for route, okind, rotated, skind, sides, n_frames, offset, families in ROUTES:
        for side in sides:
            double = "double" in (okind, skind)
            lens = _lens_cycle(k, double)
            n_src, n_out = SAMPLES[k % len(SAMPLES)], SAMPLES[(k + 2) % len(SAMPLES)]
            if lens == "nan80":  # (samples at 90 degrees and beyond are NaN: a coarse table of it is all NaN)
                n_src, n_out = max(n_src, 17), max(n_out, 17)
            k += 1
            cid = f"{route}-{okind}{'-rot' if rotated else ''}<-{skind}-{side}-{lens}-{n_out}/{n_src}"
            cases.append(pytest.param(okind, rotated, skind, side, lens, n_out, n_src, n_frames, offset, families,
                                      id=cid))
    return cases


def _case(okind, rotated, skind, side, lens, n_out, n_src, **kw):
    olens = lens if side in ("output", "both") else None
    slens = (_lens_cycle(list(LENSES).index(lens) + 1, True) if side == "both" and skind == "double" else lens) \
        if side in ("source", "both") else None
    return Case(okind, olens, ROT if rotated else (), skind, slens, n_out, n_src, **kw)


@pytest.mark.parametrize("okind,rotated,skind,side,lens,n_out,n_src,n_frames,offset,families", _route_cases())
def test_fused_routes_follow_the_table_oracle(torch_cuda, okind, rotated, skind, side, lens, n_out, n_src, n_frames,
                                              offset, families):
    torch = torch_cuda
    case = _case(okind, rotated, skind, side, lens, n_out, n_src)
    frames = _frames(case.src_shape, n_frames, seed=n_out + n_src + n_frames)
    dev = torch.from_numpy(frames).cuda()
    if offset:
        buf = torch.empty(dev.numel() + 1, dtype=torch.uint8, device="cuda")
        dev = buf[1:].view(dev.shape)
        dev.copy_(torch.from_numpy(frames).cuda())
    got, ran = case.run(dev if n_frames > 1 else dev[0])
    assert ran and set(ran) <= families, (case.cid, ran)
    print(f"{case.cid}: {sorted(ran)}")
    assert got.any(), case.cid  # (not a table that blacks out every pixel)
    case.check(got if n_frames > 1 else got[None], frames)


# ------------------------------------------------------------------------------------ row bands

@pytest.mark.parametrize("side", ["source", "output", "both"])
def test_row_bands(torch_cuda, side):
    """remap_row_band: a tile-aligned band and an odd one, each against the oracle's rows"""
    from photonbend_b200 import engine

    torch = torch_cuda
    okind, skind = ("equirect", "camera") if side == "source" else ("camera", "double" if side == "both" else "equirect")
    case = _case(okind, False, skind, side, {"source": "wavy", "output": "mismatched", "both": "kb"}[side], 3, 17)
    frame = _frames(case.src_shape, 1, seed=5)[0]
    oracle = case.oracle()
    want_families = {(64, 128): {"tiled_sep"} if side == "source" else {"direct"}, (37, 101): {"direct"}}
    with torch.no_grad():
        src = torch.from_numpy(frame).cuda()
        rays, geom = case.cmap().rays, case.src_img._source_geometry()
        full = np.zeros(oracle.cmap.shape[:2] + (3,), np.uint8)
        for band, families in want_families.items():
            got, ran = helpers.remap_launches(lambda: engine.remap_rows_device(rays, geom, src, *band))
            assert set(ran) == families, (case.cid, band, ran)
            full[band[0]:band[1]] = got.cpu().numpy()
            print(f"{case.cid} rows {band}: {sorted(ran)}")
    # the oracle's whole frame, compared on the rows the bands wrote
    want_mask = np.zeros(full.shape[:2], bool)
    for b0, b1 in want_families:
        want_mask[b0:b1] = True
    from oracle import numpy_port

    want = numpy_port.sample(case.sg, frame, oracle.cmap.copy())
    stable = helpers.stable_pixel_mask(case.sg, frame, oracle.cmap)
    if oracle.fov_edge is not None:
        stable &= ~oracle.fov_edge
    bad = (full != want).any(axis=2) & want_mask & stable
    if case.sg["kind"] == "double":
        delta = np.abs(full.astype(np.int16) - want.astype(np.int16)).max(axis=2)
        bad &= ~((delta == 1) & oracle.blended)
    assert not bad.any(), (case.cid, int(bad.sum()))


# ------------------------------------------------------------------------------------ wider elements

WIDE = [
    ("float32", 3, "equirect", False, "camera", "source"),    # separable tables through remap_wide_kernel
    ("float16", 4, "equirect", True, "camera", "source"),     # per-pixel cascade
    ("float32", 1, "camera", False, "equirect", "output"),
    ("uint16", 3, "camera", True, "camera", "both"),
]


@pytest.mark.parametrize("dtype,channels,okind,rotated,skind,side", WIDE, ids=[f"{w[0]}x{w[1]}-{w[5]}" for w in WIDE])
def test_wide_elements(torch_cuda, dtype, channels, okind, rotated, skind, side):
    torch = torch_cuda
    lens = {"source": "kb", "output": "wavy", "both": "mismatched"}[side]
    case = _case(okind, rotated, skind, side, lens, 17, 2 if side == "both" else 1025, channels=channels)
    frames = _frames(case.src_shape, 3, seed=channels, dtype=np.dtype(dtype))
    got, ran = case.run(torch.from_numpy(frames).cuda())
    assert ran == {"wide": 1}, (case.cid, ran)
    case.check(got, frames, dtype)


# ------------------------------------------------------------------------------------ typed blend

@pytest.mark.parametrize("dtype", ["uint16", "float32", "int8"])
@pytest.mark.parametrize("rotated", [False, True])
def test_keep_dtype_double_source(torch_cuda, dtype, rotated):
    """remap_blend_kernel with a table on the double source, against typed_oracle.sample_double"""
    torch = torch_cuda
    case = _case("equirect", rotated, "double", "source", "kb" if rotated else "wavy", 17, 17 if rotated else 65537,
                 keep_dtype=True)
    from photonbend_b200 import engine

    base = _frames(case.src_shape, 3, seed=31)
    scale, shift = {"uint16": (251.0, 7.0), "float32": (97.5, -3000.0)}.get(dtype, (1.0, 0.0))
    frames = (base.astype(np.float64) * scale + shift).astype(dtype) if dtype != "int8" else base.view(np.int8)
    got, ran = case.run(torch.from_numpy(np.ascontiguousarray(frames)).cuda())
    assert ran == {"blend": 1}, (case.cid, ran)
    # as tests/test_gpu_double_dtypes.py: the oracle runs on the map the device materialises, so the
    # blend weights are the kernel's bit for bit; the picks are compared where they are stable
    m = engine.materialize_map_device(case.cmap().rays).cpu().numpy()
    for k in range(len(frames)):
        want = typed_oracle.sample_double(case.sg, frames[k], m.copy(), dtype)
        stable = helpers.stable_pixel_mask(case.sg, base[k], m)
        diff = (_bytes(got[k]) != _bytes(want)).any(axis=2)
        assert not (diff & stable).any() and stable.mean() > 0.9, (case.cid, k, int((diff & stable).sum()))


# ------------------------------------------------------------------------------------ frames kernel

@pytest.mark.parametrize("dtype", ["uint8", "float32"])
@pytest.mark.parametrize("side", ["source", "output", "both"])
def test_frame_rotations(torch_cuda, dtype, side):
    """remap_frames_device: frame k against the table oracle with the rotations + (pyr_k,)"""
    from photonbend_b200 import engine
    from photonbend_b200.core.rotation import Rotation

    torch = torch_cuda
    okind, skind = {"source": ("equirect", "camera"), "output": ("camera", "equirect"), "both": ("double", "camera")}[side]
    case = _case(okind, False, skind, side, {"source": "nan80", "output": "kb", "both": "mismatched"}[side], 1025, 17)
    frames = _frames(case.src_shape, 4, seed=17, dtype=np.dtype(dtype))
    rng = np.random.default_rng(4)
    pyrs = [(0.0, math.pi, 0.0), (0.0, 0.0, 0.0)] + [tuple(rng.uniform(-3, 3, 3)) for _ in range(2)]
    mats = [Rotation(*p).rotation_matrix for p in pyrs]
    got, ran = helpers.remap_launches(lambda: engine.remap_frames_device(
        case.cmap().rays, case.src_img._source_geometry(), torch.from_numpy(frames).cuda(), mats))
    assert ran == {"frames": 1}, ran
    got = got.cpu().numpy()
    assert all(got[k].any() for k in range(len(pyrs))), case.cid
    for k, pyr in enumerate(pyrs):
        oracle = helpers.Oracle(case.og, case.rots + (pyr,), case.sg)
        oracle.check(_bytes(got[k]), _bytes(frames[k]), (case.cid, k))


# ------------------------------------------------------------------------------------ explicit maps

@pytest.mark.parametrize("lens,n", [("kb", 2), ("wavy", 17), ("nan80", 65537), ("mismatched", 1025)])
def test_explicit_maps(torch_cuda, lens, n):
    """The materialised map of a table output (latitude bit-exact, longitude to atan2's ulps), the
    gathers from a table source along the oracle's map (u8, px, typed) and map_projection of it"""
    from oracle import numpy_port
    from photonbend_b200 import engine
    from photonbend_b200.core.projection import map_projection

    torch = torch_cuda
    case = _case("camera", False, "camera", "both", lens, n, SAMPLES[(SAMPLES.index(n) + 1) % len(SAMPLES)])
    got_map, ran = helpers.remap_launches(lambda: engine.materialize_map_device(case.cmap().rays).cpu().numpy())
    assert ran == {"map": 1}, ran
    want_map = helpers.oracle_map(case.og, ())
    assert np.array_equal(got_map[:, :, 2], want_map[:, :, 2])
    assert np.array_equal(got_map[:, :, 0], want_map[:, :, 0], equal_nan=True)
    lon_ok = np.abs(got_map[:, :, 1] - want_map[:, :, 1]) <= 2 * np.spacing(np.pi)
    assert np.all(lon_ok | (np.isnan(got_map[:, :, 1]) & np.isnan(want_map[:, :, 1])))

    # gathers along the oracle's own map
    cmap = want_map
    dev_map = torch.from_numpy(cmap.copy()).cuda()
    frame = _frames(case.src_shape, 1, seed=n)[0]
    for what, arr, families in (("u8", frame, {"gather"}),
                                ("px", frame.astype(np.float32), {"gather"})):
        got, ran = helpers.remap_launches(lambda: engine.gather_from_map_device(
            case.src_img._source_geometry(), dev_map, torch.from_numpy(arr).cuda()).cpu().numpy())
        assert set(ran) == families, (what, ran)
        helpers.Oracle(case.og, (), case.sg).check(_bytes(got), _bytes(arr), (case.cid, what))
    # typed: a double source blended in uint16 along the same map
    dbl = _case("camera", False, "double", "source", lens if LENSES[lens][3] else "kb", n, n, keep_dtype=True)
    arr = (_frames(dbl.src_shape, 1, seed=3)[0].astype(np.uint16) * 251)
    got, ran = helpers.remap_launches(lambda: engine.gather_from_map_device(
        dbl.src_img._source_geometry(), dev_map, torch.from_numpy(arr).cuda()).cpu().numpy())
    assert set(ran) == {"gather"}, ran
    want = typed_oracle.sample_double(dbl.sg, arr, cmap.copy(), "uint16")
    stable = helpers.stable_pixel_mask(dbl.sg, (arr // 251).astype(np.uint8), cmap)
    diff = (got != want).any(axis=2) & stable  # (the map is the oracle's: the weights are too)
    assert not diff.any() and stable.mean() > 0.9, int(diff.sum())
    # map_projection of the materialised table map
    vis, ran = helpers.remap_launches(lambda: map_projection(case.cmap()))
    assert set(ran) <= {"map"}, ran
    with np.errstate(invalid="ignore"):  # (the NaN latitudes of a lens that is NaN past 80 degrees)
        want_vis = numpy_port.map_projection(want_map.copy())
    d = np.abs(vis.astype(np.int16) - want_vis.astype(np.int16))
    assert np.array_equal(vis[:, :, 0], want_vis[:, :, 0]) and np.array_equal(vis[:, :, 2], want_vis[:, :, 2])
    assert np.minimum(d[:, :, 1], 256 - d[:, :, 1]).max() <= 1


# ------------------------------------------------------------------------------------ raw ABI


def _desc(og, sg, channels=3):
    """pb_remap_desc of an un-rotated panorama output of a camera source with raw tables"""
    from photonbend_b200 import _native

    d = _native.RemapDesc()
    d.out.kind, d.out.height, d.out.width = _native.KIND_EQUIRECT, og["height"], og["width"]
    d.src.kind, d.src.lens, d.src.height, d.src.width = _native.KIND_CAMERA, _native.LENS_TABLE, sg["height"], sg["width"]
    d.src.fov, d.src.f_distance = sg["fov"], sg["magnitude"] / sg["lens"].forward(sg["fov"] / 2)
    table, x_max = sg["lens"].source
    d.src.lens_table = table.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    d.src.lens_table_n, d.src.lens_table_max = table.size, x_max
    d.channels = channels
    return d


def _raw_geom(table, x_max, fwd=_kb, fov=rad(200), h=240, w=256):
    lens = table_oracle.TableLens(fwd, None, (np.ascontiguousarray(table, dtype=np.float64), x_max))
    return {"kind": "camera", "height": h, "width": w, "lens": lens, "fov": fov, "magnitude": 119.5}


def _raw_run(torch, desc, frame, plan=True):
    from photonbend_b200 import _native

    lib = _native.load()
    src = torch.from_numpy(frame).cuda()
    dst = torch.empty((desc.out.height, desc.out.width, 3), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    if plan:
        handle = ctypes.c_void_p()
        _native.check(lib.pb_plan_create(ctypes.byref(desc), stream, ctypes.byref(handle)))
        try:
            _native.check(lib.pb_plan_remap_u8(handle, src.data_ptr(), 0, dst.data_ptr(), 0, 1, stream))
            torch.cuda.synchronize()
        finally:
            lib.pb_plan_destroy(handle)
    else:
        _native.check(lib.pb_remap_u8(ctypes.byref(desc), src.data_ptr(), 0, dst.data_ptr(), 0, 1, stream))
    return dst


PANO = {"kind": "equirect", "height": OUT_H, "width": OUT_W}


@pytest.mark.parametrize("plan", [True, False], ids=["plan", "planless"])
def test_raw_tables_clamp_and_special_samples(torch_cuda, plan):
    """A source table shorter than the latitudes reached (pixels past it take the last sample, the
    documented clamp), tables with negative and infinite samples, and one of 2^24 samples"""
    torch = torch_cuda
    frame = _frames((240, 256, 3), 1, seed=8)[0]
    tables = {}
    x_max = rad(70)  # latitudes up to 100 degrees reach the image: past 70 the clamp
    tables["clamped"] = (_kb(np.linspace(0, x_max, 257)), x_max)
    special = _kb(np.linspace(0, np.pi, 33))
    special[3] = -0.25
    special[20] = np.inf
    special[21] = -np.inf
    tables["negative-inf"] = (special, np.pi)
    tables["2^24"] = (_kb(np.linspace(0, np.pi, 1 << 24)), np.pi)
    for name, (table, tmax) in tables.items():
        sg = _raw_geom(table, tmax)
        desc = _desc(PANO, sg)
        got, ran = helpers.remap_launches(lambda: _raw_run(torch, desc, frame, plan).cpu().numpy())
        assert set(ran) <= {"sep1", "direct", "generic", "tiled_sep"} and ran, (name, ran)
        helpers.Oracle(PANO, (), sg).check(got, frame, (name, plan))
        if name == "clamped":  # the clamp is reached, and it is not the function
            cmap = helpers.oracle_map(PANO, ())
            assert (cmap[:, :, 0] > x_max).any()


def test_planless_call_copies_the_table_before_it_returns(torch_cuda):
    """pb_remap_u8 with a table the caller overwrites right after the call (before synchronising):
    the output follows the table as it was during the call"""
    from photonbend_b200 import _native

    torch = torch_cuda
    lib = _native.load()
    frame = _frames((240, 256, 3), 1, seed=9)[0]
    table = _kb(np.linspace(0, np.pi, 4097))
    sg = _raw_geom(table.copy(), np.pi)
    desc = _desc(PANO, sg)
    host = np.ascontiguousarray(table)  # the descriptor points here
    desc.src.lens_table = host.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    src = torch.from_numpy(frame).cuda()
    dst = torch.empty((OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _native.check(lib.pb_remap_u8(ctypes.byref(desc), src.data_ptr(), 0, dst.data_ptr(), 0, 1, stream))
    host[:] = 0.0  # every pixel would read the centre if this reached the kernel
    torch.cuda.synchronize()
    helpers.Oracle(PANO, (), sg).check(dst.cpu().numpy(), frame, "overwritten after the call")


def test_plan_cache_keys_on_the_table(torch_cuda):
    """One geometry through two different tables, one after the other: the second call follows its
    own table (engine._desc_key digests the samples, not the host pointer)"""
    torch = torch_cuda
    from photonbend_b200.core.lens import Lens
    from photonbend_b200.core.projection import CameraImage, PanoramaImage

    frame = _frames((240, 256, 3), 1, seed=10)[0]
    dev = torch.from_numpy(frame).cuda()
    cmap = PanoramaImage(np.zeros((OUT_H, OUT_W, 3), np.uint8)).get_coordinate_map()
    half = rad(200) / 2
    # the second forward function equals the first at fov / 2: same focal distance, same descriptor
    # bytes, other samples
    lenses = (Lens(_kb, _kb_inverse), Lens(lambda t: _kb(t) + 0.3 * np.sin(3 * t) * (t - half) ** 2, _kb_inverse))
    outs, keys = [], []
    for lens in lenses:
        image = CameraImage(dev, rad(200), lens, magnitude=119.5)
        _with_samples(17, image._source_geometry)
        got, ran = helpers.remap_launches(lambda: image.process_coordinate_map(cmap).cpu().numpy())
        assert ran == {"sep1": 1}, ran
        helpers.Oracle(PANO, (), table_oracle.geom_of(image)).check(got, frame, "plan cache")
        outs.append(got)
        keys.append(image.f_distance)
    assert keys[0] == keys[1] and not np.array_equal(outs[0], outs[1])
