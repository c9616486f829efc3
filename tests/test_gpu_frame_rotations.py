"""A rotation per frame (pb_plan_remap_frames_px, remap_frames_kernel): frame k of a batch must be the
bytes the plan path gives for the plan's rotations followed by M_k, on every image-kind pair and
element width, through graphs, pipelines, file streams and the directory commands."""

import ctypes
import math

import numpy as np
import pytest

import case_matrix
import helpers
import table_oracle

pytestmark = pytest.mark.gpu

rad = case_matrix.rad
F = 128  # kFramesPerLaunch (csrc/pb_frames.cuh): frames per launch
OUT_H, OUT_W = 170, 336  # partial tiles on the right and bottom edges
KINDS = ("camera", "double", "equirect")
ROTATION_SETS = ((), ((0.3, -0.2, 1.0),), ((rad(-90), 0.0, rad(195)), (0.1, 0.2, 0.3)))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _out_geom(kind):
    if kind == "equirect":
        return {"kind": "equirect", "height": OUT_H, "width": OUT_W}
    if kind == "camera":
        return {"kind": "camera", "height": OUT_H, "width": OUT_W, "lens": "equisolid", "fov": rad(180),
                "magnitude": 150.5}
    return {"kind": "double", "height": OUT_H, "width": OUT_W, "lens": "equidistant", "fov": rad(195)}


def _src_geom(kind):
    if kind == "equirect":
        return {"kind": "equirect", "height": 192, "width": 384}
    if kind == "camera":
        return {"kind": "camera", "height": 240, "width": 256, "lens": "stereographic", "fov": rad(200),
                "magnitude": 119.5}
    return {"kind": "double", "height": 192, "width": 384, "lens": "thoby", "fov": rad(190)}


def _matrices(n, seed):
    """n distinct rotations: a 180-degree yaw, the identity, then seeded ones."""
    from photonbend_b200.core.rotation import Rotation

    rng = np.random.default_rng(seed)
    mats = [Rotation(0.0, math.pi, 0.0).rotation_matrix, np.eye(3)]
    mats += [Rotation(*rng.uniform(-math.pi, math.pi, 3)).rotation_matrix for _ in range(max(0, n - 2))]
    return np.stack(mats[:n])


def _user_source(sg, shape):
    """a camera source of sg's geometry with equisolid as a Lens of user callables: PB_LENS_TABLE"""
    from photonbend_b200.core.lens import Lens
    from photonbend_b200.core.projection import CameraImage

    lens = Lens(lambda t: 2 * np.sin(t / 2), lambda r: 2 * np.arcsin(r / 2))
    return CameraImage(np.zeros(shape, np.uint8), sg["fov"], lens, magnitude=sg.get("magnitude"))


def _rays_geom(og, rots, sg, shape, user_lens=False):
    src = _user_source(sg, shape) if user_lens else helpers.product_image(sg, np.zeros(shape, np.uint8))
    return helpers.product_map(og, rots).rays, src._source_geometry()


def _check_table_oracle(got, frames, og, rots, sg, mats, what):
    """frame k of a user-lens remap against the table oracle of the map rotated by mats[k] (any 9
    doubles: numpy_port.rotate_map is the reference's arithmetic, orthonormal or not)"""
    from oracle import numpy_port

    got = got.cpu().numpy()
    with table_oracle.patched():
        for k, m in enumerate(mats):
            oracle = helpers.Oracle(og, rots, sg)
            oracle.cmap = numpy_port.rotate_map(oracle.cmap, np.asarray(m, dtype=np.float64))
            oracle.check(got[k], frames[k], f"{what}: frame {k}")


def _per_frame(torch, rays, geom, src_dev, mats, stride0=False):
    """The oracle of this file: frame k through a plan of rays + (M_k,), one frame per call."""
    from photonbend_b200 import engine

    return torch.stack([engine.remap_device(rays.rotated(m), geom, src_dev if stride0 else src_dev[k])
                        for k, m in enumerate(mats)])


def _assert_frames_equal(got, want, what):
    got, want = got.cpu(), want.cpu()
    assert got.shape == want.shape, what
    for k in range(got.shape[0]):
        assert torch_equal_bytes(got[k], want[k]), f"{what}: frame {k}"


def torch_equal_bytes(a, b):
    return np.array_equal(a.contiguous().view(-1).numpy().view(np.uint8), b.contiguous().view(-1).numpy().view(np.uint8))


# ------------------------------------------------------------------------------------ 1. kind pairs


@pytest.mark.parametrize("n", [1, 3, 2 * F + 1])
@pytest.mark.parametrize("rset", range(len(ROTATION_SETS)))
@pytest.mark.parametrize("okind", KINDS)
@pytest.mark.parametrize("skind", KINDS)
def test_every_kind_pair_matches_the_plan_path(torch_cuda, okind, skind, rset, n):
    from photonbend_b200 import engine

    torch = torch_cuda
    og, sg, rots = _out_geom(okind), _src_geom(skind), ROTATION_SETS[rset]
    shape = (sg["height"], sg["width"], 3)
    rays, geom = _rays_geom(og, rots, sg, shape)
    rng = np.random.default_rng(100 * rset + n)
    src = torch.from_numpy(rng.integers(0, 256, (n,) + shape, dtype=np.uint8)).cuda()
    if n > 1:
        src[1] = 200  # a flat frame: the double-fisheye blend on its truncation boundaries
    mats = _matrices(n, 7 + rset)
    got, ran = helpers.remap_launches(lambda: engine.remap_frames_device(rays, geom, src, mats))
    assert ran == {"frames": -(-n // F)}, ran
    _assert_frames_equal(got, _per_frame(torch, rays, geom, src, mats), f"{okind} <- {skind} {rots} n={n}")


# ------------------------------------------------------------------------------------ 2. element widths


@pytest.mark.parametrize("dtype, channels", [("uint16", 3), ("float16", 4), ("float32", 1), ("float64", 3),
                                             ("uint8", 1), ("uint8", 4), ("int32", 2)])
@pytest.mark.parametrize("skind", ["camera", "equirect"])
def test_element_widths_match_the_plan_path(torch_cuda, dtype, channels, skind):
    from photonbend_b200 import engine

    torch = torch_cuda
    og, sg = _out_geom("camera" if skind == "equirect" else "equirect"), _src_geom(skind)
    shape = (sg["height"], sg["width"], channels)
    rays, geom = _rays_geom(og, ROTATION_SETS[1], sg, shape)
    n = 5
    rng = np.random.default_rng(3)
    bits = rng.integers(0, 256, (n,) + shape + (np.dtype(dtype).itemsize,), dtype=np.uint8)
    frames = bits.view(dtype).reshape((n,) + shape)
    if np.dtype(dtype).kind == "f":  # NaN payloads and -0.0 must pass through as bytes
        frames = frames.copy()
        frames[:, ::7, ::5] = np.array(-0.0, dtype)
        nan = np.array(np.nan, dtype).view(f"u{np.dtype(dtype).itemsize}") | 5
        frames.view(f"u{np.dtype(dtype).itemsize}")[:, 3::11, 1::3] = nan
    src = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    mats = _matrices(n, 11)
    got = engine.remap_frames_device(rays, geom, src, mats)
    assert got.dtype == src.dtype
    _assert_frames_equal(got, _per_frame(torch, rays, geom, src, mats), f"{dtype} x {channels} <- {skind}")
    # a double-fisheye source takes uint8 only
    if skind == "camera" and dtype != "uint8":
        drays, dgeom = _rays_geom(og, (), _src_geom("double"), (192, 384, channels))
        with pytest.raises(NotImplementedError, match="double-fisheye source must be uint8"):
            engine.remap_frames_device(drays, dgeom, torch.zeros((1, 192, 384, channels), dtype=src.dtype,
                                                                 device="cuda"), mats[:1])


# ------------------------------------------------------------------------------------ 3. special frames


def test_non_orthonormal_frame_lens_table_and_stride_zero(torch_cuda):
    from photonbend_b200 import engine

    torch = torch_cuda
    og, sg = _out_geom("equirect"), _src_geom("camera")
    sg = dict(sg, lens="equisolid", fov=rad(180))
    shape = (sg["height"], sg["width"], 3)
    rng = np.random.default_rng(5)
    mats = _matrices(7, 13)
    mats[3] = mats[3] * 1.01            # not orthonormal: the exact chain, for this frame only
    mats[4] = np.array([[1.0, 0.2, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])  # a shear
    mats[5, 1, 1] = np.nan              # not finite
    one = torch.from_numpy(rng.integers(0, 256, shape, dtype=np.uint8)).cuda()
    batch = torch.from_numpy(rng.integers(0, 256, (7,) + shape, dtype=np.uint8)).cuda()
    for user_lens in (False, True):
        for rots in ROTATION_SETS[:2]:
            rays, geom = _rays_geom(og, rots, sg, shape, user_lens)
            what = f"user lens {user_lens} {rots}"
            got = engine.remap_frames_device(rays, geom, batch, mats)
            _assert_frames_equal(got, _per_frame(torch, rays, geom, batch, mats), what)
            if user_lens:
                sg_table = table_oracle.geom_of(_user_source(sg, shape))
                _check_table_oracle(got, batch.cpu().numpy(), og, rots, sg_table, mats, what)
            # source stride 0: seven views of one image
            _assert_frames_equal(engine.remap_frames_device(rays, geom, one, mats),
                                 _per_frame(torch, rays, geom, one, mats, stride0=True), what + " stride 0")
    # a lens table on the output side
    from photonbend_b200.core.lens import Lens
    from photonbend_b200.core.projection import CameraImage, PanoramaImage

    lens = Lens(lambda t: 2 * np.sin(t / 2), lambda r: 2 * np.arcsin(r / 2))
    out_image = CameraImage(np.zeros((OUT_H, OUT_W, 3), np.uint8), rad(180), lens, magnitude=150.5)
    rays = out_image.get_coordinate_map().rays
    geom = PanoramaImage(np.zeros((192, 384, 3), np.uint8))._source_geometry()
    pano = torch.from_numpy(rng.integers(0, 256, (7, 192, 384, 3), dtype=np.uint8)).cuda()
    got = engine.remap_frames_device(rays, geom, pano, mats)
    _assert_frames_equal(got, _per_frame(torch, rays, geom, pano, mats), "output lens table")
    _check_table_oracle(got, pano.cpu().numpy(), table_oracle.geom_of(out_image), (), _src_geom("equirect"), mats,
                        "output lens table")


# ------------------------------------------------------------------------------------ 4. NumPy oracle


def test_frames_match_the_numpy_oracle(torch_cuda):
    """Frame k against oracle/numpy_port.py with rotations + (pyr_k,), with the acceptance of
    tests/test_gpu_parity.py::test_random_mid_size_geometries."""
    from oracle import numpy_port
    from photonbend_b200 import engine
    from photonbend_b200.core.rotation import Rotation

    torch = torch_cuda
    rng = np.random.default_rng(21)
    n_px = n_bad = 0
    for okind, skind, rset in (("equirect", "double", 0), ("camera", "equirect", 1), ("double", "camera", 2),
                               ("equirect", "camera", 1)):
        og, sg, rots = _out_geom(okind), _src_geom(skind), ROTATION_SETS[rset]
        pyrs = [tuple(float(v) for v in rng.uniform(-0.3, 0.3, 3)) for _ in range(3)]
        frames = np.stack([case_matrix.case_image(sg, 900 + k) for k in range(3)])
        rays, geom = _rays_geom(og, rots, sg, frames.shape[1:])
        got = engine.remap_frames_device(rays, geom, torch.from_numpy(frames).cuda(),
                                         [Rotation(*p) for p in pyrs]).cpu().numpy()
        for k, pyr in enumerate(pyrs):
            want = numpy_port.remap(og, rots + (pyr,), sg, frames[k])
            cid = f"{og} {rots + (pyr,)} {sg}"
            assert got[k].shape == want.shape, cid
            n_px += want.shape[0] * want.shape[1]
            if np.array_equal(got[k], want):
                continue
            diff = (got[k] != want).any(axis=2)
            stable = helpers.stable_pixel_mask(sg, frames[k], numpy_port.coordinate_map(og, rots + (pyr,)))
            hard = diff & stable
            if hard.any():
                delta = np.abs(got[k].astype(np.int16) - want.astype(np.int16)).max(axis=2)
                assert sg["kind"] == "double" and delta[hard].max() == 1 and hard.mean() <= 2e-4, (cid, int(hard.sum()))
            n_bad += int(diff.sum())
    assert n_bad / n_px <= 1e-4, (n_bad, n_px)


# ------------------------------------------------------------------------------------ 5, 6. census, graphs


def test_launch_census_and_cuda_graph_capture(torch_cuda):
    from photonbend_b200 import _native, engine

    torch = torch_cuda
    og, sg = _out_geom("camera"), _src_geom("equirect")
    shape = (sg["height"], sg["width"], 3)
    rays, geom = _rays_geom(og, ROTATION_SETS[1], sg, shape)
    rng = np.random.default_rng(8)
    n = 2 * F + 3
    src = torch.from_numpy(rng.integers(0, 256, (n,) + shape, dtype=np.uint8)).cuda()
    mats = _matrices(n, 17)
    first = engine.remap_frames_device(rays, geom, src, mats)  # creates the plan
    torch.cuda.synchronize()
    before = _native.launch_counts()
    again = engine.remap_frames_device(rays, geom, src, mats)
    after = _native.launch_counts()
    delta = {k: after[k] - before[k] for k in after if after[k] != before[k]}
    assert delta == {"frames": 3}, delta  # ceil(n / F) grids, no plan-time kernel
    _assert_frames_equal(again, first, "second call")

    # captured into a CUDA graph once the plan exists; replays give the same bytes
    out = torch.zeros_like(first)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            engine.remap_frames_device(rays, geom, src, mats, out)
    torch.cuda.current_stream().wait_stream(side)
    assert not out.any()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        _assert_frames_equal(out, first, "graph replay")
        out.zero_()


# ------------------------------------------------------------------------------------ 7. too many rotations


def test_too_many_rotations_write_nothing(torch_cuda):
    from photonbend_b200 import _native, engine

    torch = torch_cuda
    og, sg = _out_geom("equirect"), _src_geom("camera")
    shape = (sg["height"], sg["width"], 3)
    rots = tuple((0.01 * k, 0.02, -0.01 * k) for k in range(_native.PB_MAX_ROTATIONS))
    rays, geom = _rays_geom(og, rots, sg, shape)
    src = torch.zeros((2,) + shape, dtype=torch.uint8, device="cuda")
    dst = torch.full((2, OUT_H, OUT_W, 3), 77, dtype=torch.uint8, device="cuda")
    mats = _matrices(2, 1)
    with pytest.raises(_native.NativeError) as err:
        engine.remap_frames_device(rays, geom, src, mats, dst)
    assert err.value.code == _native.PB_ERR_TOO_MANY_ROTATIONS
    # the library itself, through a plan of 16 rotations
    lib = _native.load()
    desc = engine._remap_desc(rays, geom, 3)
    plan = engine._plans.get(lib, desc, 0, torch)
    m = np.ascontiguousarray(mats.reshape(-1, 9))
    rc = lib.pb_plan_remap_frames_px(plan, 1, m.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                     ctypes.c_void_p(src.data_ptr()), src[0].numel(), ctypes.c_void_p(dst.data_ptr()),
                                     dst[0].numel(), 2, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == _native.PB_ERR_TOO_MANY_ROTATIONS
    assert b"PB_MAX_ROTATIONS" in lib.pb_last_error()
    torch.cuda.synchronize()
    assert (dst == 77).all()


# ------------------------------------------------------------------------------------ 8. pipelines, files, commands


@pytest.mark.parametrize("batch", [1, 4])
def test_frame_pipeline_with_rotations(torch_cuda, batch):
    from photonbend_b200 import engine
    from photonbend_b200.batch import FramePipeline
    from photonbend_b200.core.rotation import Rotation

    torch = torch_cuda
    og, sg = _out_geom("equirect"), _src_geom("double")
    shape = (sg["height"], sg["width"], 3)
    src_img = helpers.product_image(sg, np.zeros(shape, np.uint8))
    cmap = helpers.product_map(og, ROTATION_SETS[1])
    rng = np.random.default_rng(batch)
    n = 7
    frames = [torch.from_numpy(rng.integers(0, 256, shape, dtype=np.uint8)).pin_memory() for _ in range(n)]
    outs = [torch.empty((OUT_H, OUT_W, 3), dtype=torch.uint8).pin_memory() for _ in range(n)]
    rots = [Rotation(*rng.uniform(-0.2, 0.2, 3)) for _ in range(n)]
    pipe = FramePipeline(src_img, cmap, depth=2, batch=batch)
    for f, o, r in zip(frames, outs, rots):
        pipe.submit(f, o, rotation=r)
    pipe.drain()
    with pytest.raises(ValueError, match="every frame or with none"):
        pipe.submit(frames[0], outs[0])
    geom = src_img._source_geometry()
    want = _per_frame(torch, cmap.rays, geom, torch.stack(frames).cuda(), [r.rotation_matrix for r in rots])
    _assert_frames_equal(torch.stack(outs), want, f"pipeline batch {batch}")
    plain = FramePipeline(src_img, cmap, depth=2, batch=batch)
    plain.submit(frames[0], outs[0])
    with pytest.raises(ValueError, match="every frame or with none"):
        plain.submit(frames[1], outs[1], rotation=rots[1])
    plain.drain()
    assert torch_equal_bytes(outs[0], engine.remap_device(cmap.rays, geom, frames[0].cuda()).cpu())


@pytest.mark.parametrize("codec", ["pil", "nvjpeg"])
def test_remap_files_with_rotations(torch_cuda, tmp_path, codec):
    from PIL import Image

    from photonbend_b200 import stream
    from photonbend_b200.core.rotation import Rotation

    og, sg = _out_geom("equirect"), _src_geom("camera")
    shape = (sg["height"], sg["width"], 3)
    src_img = helpers.product_image(sg, np.zeros(shape, np.uint8))
    cmap = helpers.product_map(og, ROTATION_SETS[1])
    rng = np.random.default_rng(31)
    n = 6
    suffix = ".jpg" if codec == "nvjpeg" else ".png"
    ins, outs, refs = [], [], []
    for k in range(n):
        ins.append(tmp_path / f"in{k}{suffix}")
        outs.append(tmp_path / f"out{k}{suffix}")
        refs.append(tmp_path / f"ref{k}{suffix}")
        Image.fromarray(rng.integers(0, 256, shape, dtype=np.uint8)).save(ins[-1])
    rots = [Rotation(*rng.uniform(-0.3, 0.3, 3)) for _ in range(n)]
    stats = stream.remap_files(src_img, cmap, ins, outs, batch=4, codec=codec, frame_rotations=rots)
    assert stats["codec"] == codec and stats["frames"] == n
    for k in range(n):  # the per-frame plan path through the same codec
        stream.remap_files(src_img, r_map(rots[k], cmap), [ins[k]], [refs[k]], codec=codec)
        got, want = np.asarray(Image.open(outs[k])), np.asarray(Image.open(refs[k]))
        assert np.array_equal(got, want), f"{codec} frame {k}"
    with pytest.raises(ValueError, match="5 frame rotations for 6 frames"):
        stream.remap_files(src_img, cmap, ins, outs, codec=codec, frame_rotations=rots[:5])


def r_map(rotation, cmap):
    return rotation.rotate_coordinate_map(cmap)


def test_remap_jpeg_stream_with_rotations(torch_cuda):
    import io

    from PIL import Image

    from photonbend_b200 import stream
    from photonbend_b200.core.rotation import Rotation

    og, sg = _out_geom("equirect"), _src_geom("double")
    shape = (sg["height"], sg["width"], 3)
    src_img = helpers.product_image(sg, np.zeros(shape, np.uint8))
    cmap = helpers.product_map(og, ())
    rng = np.random.default_rng(41)
    jpegs = []
    for _ in range(5):
        buf = io.BytesIO()
        Image.fromarray(rng.integers(0, 256, shape, dtype=np.uint8)).save(buf, format="JPEG")
        jpegs.append(buf.getvalue())
    rots = [Rotation(*rng.uniform(-0.3, 0.3, 3)) for _ in range(5)]
    got = stream.remap_jpeg_stream(src_img, cmap, jpegs, batch=2, frame_rotations=rots)
    for k in range(5):
        want = stream.remap_jpeg_stream(src_img, r_map(rots[k], cmap), [jpegs[k]], batch=1)[0]
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(got[k]))), np.asarray(Image.open(io.BytesIO(want)))), k


def test_cli_directory_with_frame_rotations(torch_cuda, tmp_path, monkeypatch):
    from click.testing import CliRunner
    from PIL import Image

    from photonbend_b200.core.projection import PanoramaImage
    from photonbend_b200.core.rotation import Rotation
    from photonbend_b200.scripts import commands
    from photonbend_b200.scripts.main import main
    from photonbend_b200.utils import to_radians

    monkeypatch.setenv("PHOTONBEND_B200_CODEC", "pil")
    frames_dir, out_dir = tmp_path / "frames", tmp_path / "out"
    frames_dir.mkdir()
    rng = np.random.default_rng(51)
    names = [f"f{k:02d}.png" for k in range(5)]
    pixels = [rng.integers(0, 256, (96, 96, 3), dtype=np.uint8) for _ in names]
    for name, px in zip(names, pixels):
        Image.fromarray(px).save(frames_dir / name)
    angles = [tuple(float(v) for v in rng.uniform(-20, 20, 3)) for _ in names]
    lines = ["# frame pitch yaw roll", ""] + [f"{n} {p!r} {y!r} {r!r}" for n, (p, y, r) in zip(names, angles)]
    (tmp_path / "rot.txt").write_text("\n".join(lines[::-1]) + "\n")
    res = CliRunner().invoke(main, ["make-pano", "--type", "inscribed", "--lens", "equidistant", "--fov", "200",
                                    "-r", "10", "0", "5", "--frames-per-launch", "2",
                                    "--frame-rotations", str(tmp_path / "rot.txt"), str(frames_dir), str(out_dir)])
    assert res.exit_code == 0, res.output
    for name, px, (p, y, r) in zip(names, pixels, angles):
        source = commands._photo(px, "inscribed", "equidistant", to_radians(200), commands._magnitude("inscribed", px.shape))
        cmap = PanoramaImage(np.zeros((96, 192, 3), np.uint8)).get_coordinate_map()
        cmap = Rotation(to_radians(10), to_radians(0), to_radians(5)).rotate_coordinate_map(cmap)
        cmap = Rotation(to_radians(p), to_radians(y), to_radians(r)).rotate_coordinate_map(cmap)
        want = np.asarray(source.process_coordinate_map(cmap))
        assert np.array_equal(np.asarray(Image.open(out_dir / name)), want), name
