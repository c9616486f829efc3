"""Images of any numeric element type on the device (uint16, float16 / bfloat16, float32, int32,
float64 ...).  GPU only.

The remap copies a pixel's bytes: the wide kernels must pick exactly the source pixel the
parity-tested uint8 path picks.  So the reference for a wide image of P-byte pixels is the uint8
path itself, run on the image's bytes in groups of <= 4 channels and concatenated ("byte groups").
"""

import numpy as np
import pytest

import case_matrix
import helpers

pytestmark = pytest.mark.gpu

# (dtype, channels) drawn in rotation over the cases
WIDE = (("uint16", 3), ("float16", 4), ("float32", 1), ("float32", 3), ("int32", 2), ("float64", 4))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _specials(dtype):
    """Float values that must pass through untouched: NaNs with payloads, -0.0, +-inf, denormals."""
    dt = np.dtype(dtype)
    bits = {2: np.uint16, 4: np.uint32, 8: np.uint64}[dt.itemsize]
    nbits = 8 * dt.itemsize
    mant = {2: 10, 4: 23, 8: 52}[dt.itemsize]
    exp_ones = ((1 << (nbits - 1 - mant)) - 1) << mant
    raw = [exp_ones | 1, exp_ones | (1 << (mant - 1)) | 5, (1 << (nbits - 1)) | exp_ones | 3,  # NaN payloads
           1 << (nbits - 1),                                                                 # -0.0
           exp_ones, (1 << (nbits - 1)) | exp_ones,                                          # +-inf
           1, (1 << mant) - 1, (1 << (nbits - 1)) | 7]                                       # denormals
    return np.array(raw, dtype=bits).view(dt)


def wide_image(h, w, dtype, channels, seed):
    """Random bit patterns of ``dtype`` (for floats: NaNs, infinities and denormals among them),
    with the special values planted at fixed places."""
    rng = np.random.default_rng(seed)
    e = np.dtype(dtype).itemsize
    img = rng.integers(0, 256, (h, w, channels * e), dtype=np.uint8).view(dtype).reshape(h, w, channels)
    if np.dtype(dtype).kind == "f":
        sp = _specials(dtype)
        flat = img.reshape(-1)
        flat[::7] = np.resize(sp, flat[::7].size)
    return img


def byte_groups(rays, src_geom, src_dev):
    """The uint8 path on the bytes of ``src_dev`` ((N,) H, W, C wide CUDA tensor), <= 4 bytes of
    a pixel at a time, concatenated: (..., P) uint8."""
    import torch
    from photonbend_b200 import engine

    if src_dev.dim() == 2:
        src_dev = src_dev.unsqueeze(-1)
    b = src_dev.contiguous().view(torch.uint8)  # (..., C * E)
    groups = [engine.remap_device(rays, src_geom, b[..., k:k + 4].contiguous()) for k in range(0, b.shape[-1], 4)]
    return torch.cat(groups, dim=-1)


def _as_bytes(torch, t):
    t = t if t.dim() != 2 else t.unsqueeze(-1)
    return t.contiguous().view(torch.uint8)


def _check_against_groups(torch, rays, src_geom, src_dev, got_dev, what):
    want = byte_groups(rays, src_geom, src_dev)
    got = _as_bytes(torch, got_dev).reshape(want.shape)
    bad = (got != want).reshape(-1, want.shape[-1]).any(dim=1)
    assert int(bad.sum()) == 0, (what, int(bad.sum()))


def test_every_non_double_case_picks_the_uint8_path_pixels(torch_cuda):
    """1215 cases of the parity matrix (every case whose source is not a double fisheye)."""
    torch = torch_cuda
    n = 0
    for k, (cid, og, rots, sg, seed) in enumerate(c for c in case_matrix.all_cases() if c[3]["kind"] != "double"):
        dtype, channels = WIDE[k % len(WIDE)]
        image = wide_image(sg["height"], sg["width"], dtype, channels, seed)
        got = helpers.product_remap(og, rots, sg, image)
        assert isinstance(got, np.ndarray) and got.dtype == image.dtype, cid
        cmap = helpers.product_map(og, rots)
        src_geom = helpers.product_image(sg, image)._source_geometry()
        want = byte_groups(cmap.rays, src_geom, torch.from_numpy(image).cuda()).cpu().numpy()
        diff = (got.view(np.uint8).reshape(want.shape) != want).any(axis=-1)
        assert int(diff.sum()) == 0, (cid, dtype, channels, int(diff.sum()))
        n += 1
    assert n == 1215


def test_golden_cases_agree_with_the_reference_oracle(torch_cuda, golden_small):
    """The NumPy oracle (bit-identical to the reference) on the same wide image, with the stable-pixel
    allowance the uint8 parity tests apply (helpers.stable_pixel_mask, on the image's bytes)."""
    from oracle import numpy_port
    from test_gpu_parity import BY_ID, MAX_DEGENERATE_GOLDEN

    _, outputs, _ = golden_small
    n_px = n_boundary = n_degenerate = n_cases = 0
    for k, key in enumerate(sorted({"__".join(f.split("__")[:3]) for f in outputs.files})):
        _, og, rots, sg, seed = BY_ID[key]
        if sg["kind"] == "double":
            continue
        dtype, channels = WIDE[k % len(WIDE)]
        image = wide_image(sg["height"], sg["width"], dtype, channels, seed)
        got = helpers.product_remap(og, rots, sg, image)
        want = numpy_port.remap(og, rots, sg, image)
        assert got.dtype == want.dtype == image.dtype and got.shape == want.shape, key
        gb = got.view(np.uint8).reshape(got.shape[0], got.shape[1], -1)
        wb = want.view(np.uint8).reshape(gb.shape)
        n_cases += 1
        diff = (gb != wb).any(axis=2)
        if not diff.any():
            n_px += diff.size
            continue
        stable = helpers.stable_pixel_mask(sg, image.view(np.uint8).reshape(image.shape[0], image.shape[1], -1),
                                           numpy_port.coordinate_map(og, rots))
        assert not (diff & stable).any(), (key, int((diff & stable).sum()))
        if (~stable).mean() > 0.01:
            n_degenerate += 1
        else:
            n_boundary += int(diff.sum())
            n_px += diff.size
    assert n_cases > 300
    assert n_boundary / n_px <= 1e-4, (n_boundary, n_px)
    assert n_degenerate <= MAX_DEGENERATE_GOLDEN, n_degenerate


def _full_source(torch, wl, dtype, channels, frames=None, seed=5):
    src = wl["src"]
    e = torch.empty((), dtype=dtype).element_size()
    g = torch.Generator(device="cuda").manual_seed(seed)
    shape = ((frames,) if frames else ()) + (src["height"], src["width"], channels * e)
    raw = torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
    return raw.view(dtype)


@pytest.mark.parametrize("name,dtype,channels", [("T", "float32", 3), ("cfg2", "uint16", 3), ("cfg3", "bfloat16", 3)])
def test_full_size_one_frame(torch_cuda, name, dtype, channels):
    torch = torch_cuda
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS[name]
    src = _full_source(torch, wl, getattr(torch, dtype), channels)
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    image = helpers.product_image(wl["src"], src)
    got = image.process_coordinate_map(cmap)
    assert got.is_cuda and got.dtype == src.dtype
    assert tuple(got.shape) == workloads.output_shape(wl["out"], channels)
    _check_against_groups(torch, cmap.rays, image._source_geometry(), src, got, name)


def test_full_size_batch_is_one_launch(torch_cuda):
    """T geometry, a float16 RGBA batch of 6 frames through remap_batch."""
    torch = torch_cuda
    from photonbend_b200 import _native, batch, workloads

    wl = workloads.WORKLOADS["T"]
    frames = _full_source(torch, wl, torch.float16, 4, frames=6)
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    image = helpers.product_image(wl["src"], frames[0])
    batch.remap_batch(image, cmap, frames[:2])  # the plan of this geometry exists after this call
    torch.cuda.synchronize()
    lib = _native.load()
    before = lib.pb_kernel_launches()
    got = batch.remap_batch(image, cmap, frames)
    assert lib.pb_kernel_launches() - before == 1
    assert got.dtype == torch.float16 and tuple(got.shape) == (6,) + workloads.output_shape(wl["out"], 4)
    _check_against_groups(torch, cmap.rays, image._source_geometry(), frames, got, "T x6 float16")


def test_row_bands_concatenate_to_the_frame(torch_cuda):
    torch = torch_cuda
    from photonbend_b200 import batch, workloads

    for name in ("T", "cfg3"):
        wl = workloads.WORKLOADS[name]
        src = _full_source(torch, wl, torch.float32, 3, seed=11)
        cmap = helpers.product_map(wl["out"], wl["rotations"])
        image = helpers.product_image(wl["src"], src)
        whole = image.process_coordinate_map(cmap)
        height = wl["out"]["height"]
        for world in (1, 3, 5):
            bands = [batch.remap_row_band(image, cmap, src, batch.shard_rows(height, r, world)) for r in range(world)]
            assert all(b.dtype == torch.float32 for b in bands)
            assert torch.equal(torch.cat(bands).view(torch.uint8), whole.view(torch.uint8)), (name, world)
        band = batch.remap_row_band(image, cmap, src, range(100, 333))  # off a 64-row boundary
        assert torch.equal(band.view(torch.uint8), whole[100:333].view(torch.uint8)), name


def test_explicit_maps(torch_cuda):
    """ndarray map and CUDA map equal the lazy path for float32; an equirect source zeroes the
    invalid entries of the caller's map exactly as the uint8 path does."""
    torch = torch_cuda
    cases = [c for c in case_matrix.all_cases() if c[3]["kind"] != "double"][::40]
    assert len(cases) >= 10
    for cid, og, rots, sg, seed in cases:
        image = wide_image(sg["height"], sg["width"], "float32", 3, seed)
        lazy = helpers.product_remap(og, rots, sg, image)
        src = helpers.product_image(sg, image)
        host_map = np.array(np.asarray(helpers.product_map(og, rots)), dtype=np.float64)
        u8_map = host_map.copy()
        got = src.process_coordinate_map(host_map)
        assert got.dtype == np.float32
        assert np.array_equal(got.view(np.uint32), lazy.view(np.uint32)), cid
        helpers.product_image(sg, case_matrix.case_image(sg, seed)).process_coordinate_map(u8_map)
        assert np.array_equal(host_map.view(np.uint64), u8_map.view(np.uint64)), cid  # the same side effects
        dev_map = torch.from_numpy(np.array(np.asarray(helpers.product_map(og, rots)))).cuda()
        dev_u8 = dev_map.clone()
        got_dev = src.process_coordinate_map(dev_map)
        assert np.array_equal(np.asarray(got_dev).view(np.uint32), lazy.view(np.uint32)), cid
        helpers.product_image(sg, case_matrix.case_image(sg, seed)).process_coordinate_map(dev_u8)
        assert torch.equal(dev_map.view(torch.int64), dev_u8.view(torch.int64)), cid


@pytest.mark.parametrize("batch_size", [1, 3])
def test_frame_pipeline_float16(torch_cuda, batch_size):
    torch = torch_cuda
    from photonbend_b200 import batch

    og = {"kind": "equirect", "height": 256, "width": 512}
    sg = {"kind": "camera", "height": 300, "width": 300, "lens": "equidistant", "fov": case_matrix.rad(200),
          "magnitude": 149.5}
    cmap = helpers.product_map(og, [(0.2, 0.1, -0.3)])
    frames = [torch.from_numpy(wide_image(300, 300, "float16", 4, 40 + k)).pin_memory() for k in range(5)]
    outs = [torch.empty((256, 512, 4), dtype=torch.float16).pin_memory() for _ in frames]
    image = helpers.product_image(sg, frames[0])
    pipe = batch.FramePipeline(image, cmap, depth=2, batch=batch_size)
    pipe.run(frames, outs)
    want = batch.remap_batch(image, cmap, torch.stack(frames).cuda()).cpu()
    for k, out in enumerate(outs):
        assert out.dtype == torch.float16
        assert torch.equal(out.view(torch.int16), want[k].view(torch.int16)), k


def test_flavours_alignment_and_one_byte_types(torch_cuda):
    torch = torch_cuda
    from photonbend_b200 import engine

    og = {"kind": "camera", "height": 70, "width": 90, "lens": "equisolid", "fov": case_matrix.rad(180),
          "magnitude": 35.0}
    sg = {"kind": "equirect", "height": 64, "width": 128}
    rots = [(0.3, -0.2, 1.0)]
    cmap = helpers.product_map(og, rots)
    img = wide_image(64, 128, "float32", 3, 3)
    # flavours
    got_np = helpers.product_remap(og, rots, sg, img)
    assert isinstance(got_np, np.ndarray) and got_np.dtype == np.float32
    got_cpu = helpers.product_remap(og, rots, sg, torch.from_numpy(img))
    assert engine.is_torch_tensor(got_cpu) and not got_cpu.is_cuda and got_cpu.dtype == torch.float32
    assert np.array_equal(got_cpu.numpy().view(np.uint32), got_np.view(np.uint32))
    bf = torch.from_numpy(wide_image(64, 128, "uint16", 3, 4)).cuda().view(torch.bfloat16)
    got_bf = helpers.product_remap(og, rots, sg, bf)
    assert got_bf.is_cuda and got_bf.dtype == torch.bfloat16
    _check_against_groups(torch, cmap.rays, helpers.product_image(sg, bf)._source_geometry(), bf, got_bf, "bf16")
    # views at odd element offsets (not 16-byte aligned): the same bytes
    geom = helpers.product_image(sg, img)._source_geometry()
    for dtype, channels in (("float32", 3), ("float16", 4), ("float64", 4), ("int32", 2), ("uint16", 3)):
        t = getattr(torch, dtype)
        src = torch.from_numpy(wide_image(64, 128, dtype, channels, 9)).cuda()
        aligned = engine.remap_device(cmap.rays, geom, src)
        n_src, n_out = src.numel(), aligned.numel()
        base_src = torch.empty(n_src + 1, dtype=t, device="cuda")
        base_out = torch.empty(n_out + 3, dtype=t, device="cuda")
        src_view = base_src[1:].view(src.shape)
        src_view.copy_(src)
        out_view = base_out[3:].view(aligned.shape)
        assert src_view.data_ptr() % 16 != 0 and out_view.data_ptr() % 16 != 0
        engine.remap_device(cmap.rays, geom, src_view, out_view)
        assert torch.equal(out_view.view(torch.uint8), aligned.view(torch.uint8)), dtype
    # int8 and bool through the uint8 kernels
    u8 = case_matrix.case_image(sg, 21)
    want = helpers.product_remap(og, rots, sg, u8)
    got_i8 = helpers.product_remap(og, rots, sg, u8.view(np.int8))
    assert got_i8.dtype == np.int8 and np.array_equal(got_i8.view(np.uint8), want)
    flags = (u8 & 1).astype(bool)
    got_b = helpers.product_remap(og, rots, sg, torch.from_numpy(flags).cuda())
    assert got_b.dtype == torch.bool
    assert np.array_equal(got_b.cpu().numpy(), helpers.product_remap(og, rots, sg, flags.view(np.uint8)).view(bool))


def test_wide_double_fisheye_source_is_refused(torch_cuda):
    og = {"kind": "equirect", "height": 32, "width": 64}
    sg = {"kind": "double", "height": 40, "width": 80, "lens": "equidistant", "fov": case_matrix.rad(190)}
    image = wide_image(40, 80, "float32", 3, 1)
    with pytest.raises(NotImplementedError, match="double-fisheye source must be uint8"):
        helpers.product_remap(og, [], sg, image)
