"""A double-fisheye source blended in its own dtype (DoubleCameraImage(..., keep_dtype=True)):
remap_blend_kernel for batches and row bands, the typed branches of remap_frames_kernel and
gather_from_map_kernel.  GPU only.

Every output element must be the reference's blend with its uint8 cast replaced,
``(left.astype(float64) * w_left + right.astype(float64) * w_right)`` cast as tests/typed_oracle.py:
cast_x86 says (NumPy's astype on x86-64; bfloat16: torch's cast), NaNs compared as NaNs.  The oracle
runs on the coordinate map the device materialises, so that the blend weights -- pure arithmetic on
the latitude -- are the kernel's bit for bit; which source pixel the reference picks from that map
is compared on the pixels whose pick does not hang on the last ulps of libm (helpers.stable_pixel_mask),
as the uint8 parity matrix does.
"""

import hashlib
import json
import os

import numpy as np
import pytest

import case_matrix
import helpers
import typed_oracle

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FLOATS = ("float16", "float32", "float64")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _torch_dtype(torch, name):
    return getattr(torch, "bool" if name == "bool" else name)


def double_image(sg, array):
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage

    return DoubleCameraImage(array, sg["fov"], getattr(pb_lens, sg["lens"])(), keep_dtype=True)


def frames_of(dtype, shape, seed):
    """(numpy frames the oracle reads, the same frames as a torch CPU tensor of ``dtype``): random
    values over the type's range, for floats with NaN, +-inf, -0.0 and denormals among them;
    bfloat16 frames reach the oracle as the float32 values they hold."""
    import torch

    rng = np.random.default_rng(seed)
    if dtype == "bool":
        a = rng.integers(0, 2, shape).astype(bool)
        return a, torch.from_numpy(a)
    if dtype in FLOATS or dtype == "bfloat16":
        a = (rng.standard_normal(shape) * rng.choice([1.0, 300.0, 1e5], shape)).astype(np.float32)
        flat = a.reshape(-1)
        flat[::11] = np.resize(np.array([np.nan, np.inf, -np.inf, -0.0, 1e-41, -3e-39, 6e-8, 65519.0], np.float32),
                               flat[::11].size)
        if dtype == "bfloat16":
            t = torch.from_numpy(a).to(torch.bfloat16)
            return t.float().numpy(), t
        a = a.astype(dtype)
        return a, torch.from_numpy(a)
    info = np.iinfo(dtype)
    a = rng.integers(info.min, info.max, shape, dtype=dtype, endpoint=True)
    return a, torch.from_numpy(a)


def to_numpy(torch, t, dtype):
    t = t.cpu()
    if dtype == "bfloat16":
        return t.view(torch.int16).numpy().view(np.uint16)
    return t.numpy()


def _nan_bits(b, dtype):
    if dtype == "bfloat16":
        return ((b & 0x7F80) == 0x7F80) & ((b & 0x7F) != 0)
    return np.isnan(b)


def same_px(got, want, dtype):
    """(H, W) pixels whose every element is bit-identical, a NaN counting equal to any NaN."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, want.shape, got.dtype, want.dtype)
    if dtype in FLOATS:
        bits = {2: np.uint16, 4: np.uint32, 8: np.uint64}[got.dtype.itemsize]
        ok = (got.view(bits) == want.view(bits)) | (np.isnan(got) & np.isnan(want))
    elif dtype == "bfloat16":
        ok = (got == want) | (_nan_bits(got, dtype) & _nan_bits(want, dtype))
    else:
        ok = got == want
    return ok.reshape(got.shape[0], got.shape[1], -1).all(axis=2)


def oracle(sg, frame, cmap, dtype):
    with np.errstate(all="ignore"):
        return typed_oracle.sample_double(sg, frame, cmap.copy(), dtype)


def device_map(torch, cmap):
    from photonbend_b200 import engine

    return engine.materialize_map_device(cmap.rays).cpu().numpy()


def assert_bits_equal(torch, a, b, what):
    """Two device results of one dtype: byte for byte, NaN positions equal."""
    if a.dtype.is_floating_point:
        na, nb = torch.isnan(a), torch.isnan(b)
        assert torch.equal(na, nb), what
        a, b = torch.where(na, torch.zeros_like(a), a), torch.where(nb, torch.zeros_like(b), b)
    assert torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8)), what


# ----------------------------------------------------------------------------- full size, cfg5


def _cfg5(n):
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["cfg5"]
    with open(os.path.join(GOLDEN, "cfg5_frames.json")) as fh:
        golden = json.load(fh)["frames"]
    return wl, golden, np.stack([workloads.source_image(wl, frame=k) for k in range(n)])


def test_cfg5_frames_widened_keep_their_low_bytes(torch_cuda):
    """The eight cfg5 frames widened to every integer type, through ONE remap_batch call each: every
    weight of cfg5 keeps the blend below 2^31, where every integer cast keeps the low bits of the
    same truncation as the uint8 cast -- so the low byte of each element is the reference's uint8
    output (its sha256 in tests/golden/cfg5_frames.json).  As float64 the frames blend to the very
    sums the uint8 cast truncates: cast back with that rule they give the same bytes."""
    torch = torch_cuda
    from photonbend_b200.batch import remap_batch

    n = 8
    wl, golden, frames = _cfg5(n)
    u8 = torch.from_numpy(frames).cuda()
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    for dtype in ("uint16", "int16", "int32", "uint32", "int64", "uint64", "float64"):
        batch = u8.to(_torch_dtype(torch, dtype))
        out, ran = helpers.remap_launches(lambda: remap_batch(double_image(wl["src"], batch), cmap, batch))
        assert ran == {"blend": 1}, (dtype, ran)
        assert out.dtype == batch.dtype
        if dtype == "float64":
            low = [typed_oracle.cast_x86(out[k].cpu().numpy(), "uint8") for k in range(n)]
        else:
            low = [(out[k].to(torch.int64) & 0xFF).to(torch.uint8).cpu().numpy() for k in range(n)]
        for k in range(n):
            assert hashlib.sha256(low[k].tobytes()).hexdigest() == golden[k]["out_sha256"], (dtype, k)
        del batch, out


@pytest.mark.parametrize("dtype", ["uint16", "float32"])
def test_full_size_cfg4_frame_against_the_oracle(torch_cuda, dtype):
    torch = torch_cuda
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["cfg4"]
    sg = wl["src"]
    frame, t = frames_of(dtype, (sg["height"], sg["width"], 3), 44)
    cmap = helpers.product_map(wl["out"], ())
    got = double_image(sg, t).process_coordinate_map(cmap)
    want = oracle(sg, frame, device_map(torch, cmap), dtype)
    bad = ~same_px(got, want, dtype)
    assert not bad.any(), (dtype, int(bad.sum()))


# ----------------------------------------------------------------------------- the parity matrix

MATRIX_TYPES = ("uint16", "float16", "bfloat16", "float32", "float64", "int8", "bool")


def _double_cases():
    return [c for c in case_matrix.all_cases() if c[3]["kind"] == "double"]


@pytest.mark.parametrize("dtype", MATRIX_TYPES)
def test_every_double_source_case_against_the_oracle(torch_cuda, dtype):
    """Every double-source case of the parity matrix, as a batch of two frames of one to four
    channels; bit-exact on the stable pixels, and almost all pixels stable."""
    torch = torch_cuda
    from photonbend_b200.batch import remap_batch

    checked = total = 0
    for n, (cid, og, rots, sg, seed) in enumerate(_double_cases()):
        channels = 1 + n % 4
        frames, t = frames_of(dtype, (2, sg["height"], sg["width"], channels), seed)
        cmap = helpers.product_map(og, rots)
        dev = t.cuda()
        out, ran = helpers.remap_launches(lambda: remap_batch(double_image(sg, dev), cmap, dev))
        assert ran == {"blend": 1}, (cid, ran)
        got = to_numpy(torch, out, dtype)
        m = device_map(torch, cmap)
        probe = case_matrix.case_image(sg, seed, channels)
        stable = helpers.stable_pixel_mask(sg, probe, m)
        for k in range(2):
            same = same_px(got[k], oracle(sg, frames[k], m, dtype), dtype)
            assert same[stable].all(), (cid, dtype, k, int((~same & stable).sum()))
        checked += int(stable.sum())
        total += stable.size
    assert checked >= 0.97 * total, (checked, total)


@pytest.mark.parametrize("dtype", ["float32", "uint16", "bool"])
def test_frame_rotations_match_the_plan_path(torch_cuda, dtype):
    """remap_batch(frame_rotations=...): frame k is byte for byte the plan of the map with that
    rotation appended, from a batch and from one image seen through every rotation (stride 0);
    and the oracle on the device's map of that frame."""
    torch = torch_cuda
    from photonbend_b200 import engine
    from photonbend_b200.batch import remap_batch
    from photonbend_b200.core.rotation import Rotation

    sg = {"kind": "double", "height": 40, "width": 80, "lens": "equidistant", "fov": case_matrix.rad(195)}
    rots = [Rotation(0.3 * k, -0.2 * k, 0.1 + k) for k in range(3)]
    for og in ({"kind": "equirect", "height": 32, "width": 64},
               {"kind": "camera", "height": 36, "width": 44, "lens": "equisolid", "fov": case_matrix.rad(180),
                "magnitude": 21.5}):
        cmap = helpers.product_map(og, ((0.1, 0.2, 0.3),))
        frames, t = frames_of(dtype, (3, 40, 80, 3), 9)
        dev = t.cuda()
        src = double_image(sg, dev)
        geom = src._source_geometry()
        for stride0 in (False, True):
            if stride0:  # one image seen through every rotation: source frame stride 0
                call = lambda: engine.remap_frames_device(cmap.rays, geom, dev[0], rots)  # noqa: E731
            else:
                call = lambda: remap_batch(src, cmap, dev, frame_rotations=rots)  # noqa: E731
            out, ran = helpers.remap_launches(call)
            assert ran == {"frames": 1}, ran
            for k in range(3):
                one = engine.remap_device(cmap.rays.rotated(rots[k].rotation_matrix), geom, dev[0 if stride0 else k])
                assert_bits_equal(torch, out[k], one, (og["kind"], stride0, k))
        m = device_map(torch, rots[2].rotate_coordinate_map(cmap))
        stable = helpers.stable_pixel_mask(sg, case_matrix.case_image(sg, 3), m)
        same = same_px(to_numpy(torch, out[2], dtype), oracle(sg, frames[0], m, dtype), dtype)
        assert same[stable].all() and stable.mean() > 0.9


# ----------------------------------------------------------------------------- blend edges

EDGE_FOVS = [195, 180, 181, 210, 170, 250, 180.00000000001, 179.99999999999]
NEAR_180 = [float(np.nextafter(np.pi, np.inf)), float(np.nextafter(np.pi, 0.0)), np.pi + 1e-12, np.pi - 1e-12,
            case_matrix.rad(180.000000001), np.pi, case_matrix.rad(180.0000001)]
EDGE_TYPES = ("uint16", "float32", "int32", "uint32", "int64", "uint64", "float16", "bfloat16", "float64", "int8", "bool")


def _edge_frames(h, w):
    """Flat frames on the truncation and rounding boundaries (200 w_l + 200 w_r can be
    199.99999999999997: uint16 199, float32 200.0), and frames of special values."""
    flat = [np.full((h, w, 3), v, np.float64) for v in (200.0, 1.0, 65535.0, 2.0**53 + 1.0, -0.0)]
    specials = np.resize(np.array([np.nan, np.inf, -np.inf, -0.0, 5e-324, 1e-310, 2.0**60 + 2.0**10, -1.5, 0.5]),
                         h * w * 3).reshape(h, w, 3)
    return flat + [specials, np.roll(specials, 1, axis=1)]


def _cast_frames(frames, dtype):
    import torch

    out = []
    for f in frames:
        if dtype == "bfloat16":
            t = torch.from_numpy(f).to(torch.bfloat16)
            out.append((t.float().numpy(), t))
        elif dtype == "float64":
            out.append((f, torch.from_numpy(f)))
        else:
            a = typed_oracle.cast_x86(f, dtype) if dtype not in FLOATS else f.astype(dtype)
            out.append((a, torch.from_numpy(a)))
    return out


@pytest.mark.parametrize("fov", EDGE_FOVS + NEAR_180, ids=[str(f) for f in EDGE_FOVS] + [f"near180-{k}" for k in
                                                                                           range(len(NEAR_180))])
def test_blend_edges(torch_cuda, fov):
    """Sensor fovs of the uint8 blend-band test, and those within 1e-9 rad of pi whose weights are NaN
    or run to 1e13 (uint32 beyond 2^32: NumPy's one-element cast), on flat and special-value frames,
    separable (batch) and rotated (one frame) -- every pixel, against the oracle on the same map."""
    torch = torch_cuda
    from photonbend_b200.batch import remap_batch

    fov = case_matrix.rad(fov) if fov > 10 else fov
    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": fov}
    og = {"kind": "equirect", "height": 352, "width": 704}
    base = _edge_frames(336, 672)
    for rots in ((), ((0.3, -0.7, 1.1),)):
        cmap = helpers.product_map(og, rots)
        m = device_map(torch, cmap)
        stable = np.ones((352, 704), bool) if not rots else helpers.stable_pixel_mask(
            sg, case_matrix.case_image(sg, 5), m)
        for dtype in EDGE_TYPES:
            frames = _cast_frames(base, dtype)
            batch = torch.stack([t for _, t in frames]).cuda()
            got = to_numpy(torch, remap_batch(double_image(sg, batch), cmap, batch), dtype)
            for k, (f, _) in enumerate(frames):
                same = same_px(got[k], oracle(sg, f, m, dtype), dtype)
                assert same[stable].all(), (fov, bool(rots), dtype, k, int((~same & stable).sum()))


# ----------------------------------------------------------------------------- every route agrees


@pytest.mark.parametrize("dtype", ["float32", "int64", "bfloat16", "int8"])
def test_every_route_agrees(torch_cuda, dtype):
    """Row bands concatenate to the frame; an explicit map equals the lazy one; FramePipeline gives
    the batch's frames at batch 1 and 3; a batch is ONE launch of remap_blend_kernel."""
    torch = torch_cuda
    from photonbend_b200.batch import FramePipeline, remap_batch, remap_row_band

    sg = {"kind": "double", "height": 200, "width": 400, "lens": "equisolid", "fov": case_matrix.rad(200)}
    for og, rots in (({"kind": "equirect", "height": 150, "width": 300}, ()),
                     ({"kind": "equirect", "height": 150, "width": 300}, ((0.2, 0.4, -0.3),)),
                     ({"kind": "camera", "height": 130, "width": 170, "lens": "stereographic", "fov": 2.5,
                       "magnitude": 60.0}, ((0.5, 0.1, 0.0),)),
                     ({"kind": "double", "height": 100, "width": 201, "lens": "equidistant", "fov": 3.4}, ())):
        _, t = frames_of(dtype, (4, 200, 400, 3), 21)
        dev = t.cuda()
        src = double_image(sg, dev)
        cmap = helpers.product_map(og, rots)
        out, ran = helpers.remap_launches(lambda: remap_batch(src, cmap, dev))
        assert ran == {"blend": 1}, ran
        one = double_image(sg, dev[2]).process_coordinate_map(cmap)
        assert_bits_equal(torch, out[2], one, (og["kind"], "single frame"))
        h = out.shape[1]
        bands = [remap_row_band(src, cmap, dev[1], range(a, b)) for a, b in ((0, 64), (64, 67), (67, h))]
        assert_bits_equal(torch, torch.cat(bands), out[1], (og["kind"], "bands"))
        explicit = double_image(sg, dev[3]).process_coordinate_map(torch.from_numpy(device_map(torch, cmap)).cuda())
        assert_bits_equal(torch, explicit, out[3], (og["kind"], "explicit map"))
        host_in = [dev[k].cpu() for k in range(4)]
        for batch in (1, 3):
            host_out = [torch.zeros_like(out[k], device="cpu") for k in range(4)]
            pipe = FramePipeline(double_image(sg, host_in[0]), cmap, depth=2, batch=batch)
            pipe.run(host_in, host_out)
            for k in range(4):
                assert host_out[k].dtype == t.dtype
                assert_bits_equal(torch, host_out[k].cuda(), out[k], (og["kind"], "pipeline", batch, k))


def test_uint8_with_keep_dtype_runs_the_uint8_kernels(torch_cuda):
    torch = torch_cuda
    from photonbend_b200.batch import remap_batch
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage

    sg = {"kind": "double", "height": 336, "width": 672, "lens": "equidistant", "fov": case_matrix.rad(195)}
    og = {"kind": "equirect", "height": 352, "width": 704}
    frames = torch.from_numpy(np.stack([case_matrix.case_image(sg, s) for s in (1, 2, 3)])).cuda()
    for rots in ((), ((0.3, -0.7, 1.1),)):
        cmap = helpers.product_map(og, rots)
        default, ran0 = helpers.remap_launches(
            lambda: remap_batch(DoubleCameraImage(frames, sg["fov"], pb_lens.equidistant()), cmap, frames))
        keep, ran1 = helpers.remap_launches(lambda: remap_batch(double_image(sg, frames), cmap, frames))
        assert torch.equal(default, keep) and ran0 == ran1 and "blend" not in ran1, (ran0, ran1)


# ----------------------------------------------------------------------------- past 4 GiB


def test_float64_rgba_batch_past_4_gib(torch_cuda):
    """cfg4 geometry, float64 RGBA: 944 MB per frame, six frames -- byte offsets of the last frame
    past 4 GiB in both the source and the output.  Its output must equal the remap of that frame
    alone, and the oracle on a sample of rows."""
    torch = torch_cuda
    from photonbend_b200 import workloads
    from photonbend_b200.batch import remap_batch

    wl = workloads.WORKLOADS["cfg4"]
    sg, og = wl["src"], wl["out"]
    n, shape = 6, (sg["height"], sg["width"], 4)
    frame_bytes = int(np.prod(shape)) * 8
    free, _ = torch.cuda.mem_get_info()
    if free < 3 * n * frame_bytes:
        pytest.skip(f"needs {3 * n * frame_bytes / 2**30:.1f} GiB of device memory, {free / 2**30:.1f} free")
    gen = torch.Generator(device="cuda").manual_seed(7)
    batch = (torch.rand((n,) + shape, dtype=torch.float64, device="cuda", generator=gen) * 1000.0)
    assert (n - 1) * frame_bytes >= 4 * 2**30
    cmap = helpers.product_map(og, ())
    out, ran = helpers.remap_launches(lambda: remap_batch(double_image(sg, batch), cmap, batch))
    assert ran == {"blend": 1}
    last = batch[n - 1].clone()
    alone = double_image(sg, last).process_coordinate_map(cmap)
    assert_bits_equal(torch, out[n - 1], alone, "last frame")
    rows = slice(1800, 1830)
    m = device_map(torch, cmap)[rows]
    want = oracle(sg, last.cpu().numpy(), m, "float64")
    assert same_px(out[n - 1][rows].cpu().numpy(), want, "float64").all()
