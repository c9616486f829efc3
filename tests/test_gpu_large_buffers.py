"""Sources, outputs and batches past 2 and 4 GiB, and outputs taller than a grid's 65535 rows of
blocks.

The direct, direct32, tiled and sep1 kernels form source byte offsets in 32-bit ints; plan_run keeps
them for sources of fewer than 2^31 bytes (src_pitch * H) and sends larger ones to
remap_generic_kernel.  The wide, frames and explicit-map kernels use 64-bit offsets everywhere.
Each case checks the route through the launch census and the pixels against the C oracle.

The sources never exist on the host: each is filled on the device, in row chunks, with a hash of
(linear pixel index, channel) (uint8), or with the index itself (float32).  The expected output
then follows from oracle.c_port.source_index on the geometry alone.  A pixel may differ from it
only by an index flip: the oracle's float64 coordinate sits within rounding of a pixel boundary and
the kernel took the neighbouring source pixel (see helpers.attribute_mismatches).  Double-fisheye
sources need the blend: they are checked against the NumPy oracle on a host copy, with the acceptance
of helpers.Oracle (on row bands for large outputs).

Each case frees its buffers before the next one allocates, and is skipped only when the device
cannot hold it."""

import ctypes
import time

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu

GIB = 1 << 30
OUT_H, OUT_W = 170, 336  # partial tiles on both edges; W % 4 == 0 (the direct kernels)
# the 32-bit offsets' ceiling: 3 W H < 2^31 at W = 37840 holds up to H = 18917
GUARD_W, GUARD_H = 37840, 18917
CAMERA = {"lens": "equidistant", "fov": 200 * np.pi / 180}
DOUBLE = {"lens": "equidistant", "fov": 195 * np.pi / 180}
ROT = ((0.3, -0.2, 1.0),)
_HASH_K = (1103515245, 2147483629, 1540483477)
CANARY = 0xA5


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture
def device_room(torch_cuda):
    """-> need(bytes, what): skips the test when the device cannot hold `bytes` more; frees the
    allocator's cache before and after the test, and reports the test's peak."""
    torch = torch_cuda
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()

    def need(nbytes, what):
        free, total = torch.cuda.mem_get_info()
        if free < nbytes + GIB // 2:
            pytest.skip(f"{what}: needs {nbytes / GIB:.1f} GiB of device memory, {free / GIB:.1f} GiB free of "
                        f"{total / GIB:.1f}")

    yield need
    torch.cuda.synchronize()
    print(f"peak device memory {torch.cuda.max_memory_allocated() / GIB:.2f} GiB, "
          f"{time.perf_counter() - t0:.1f} s")
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------ sources


def _geom(kind, h, w):
    if kind == "equirect":
        return {"kind": "equirect", "height": h, "width": w}
    return dict({"kind": kind, "height": h, "width": w}, **(CAMERA if kind == "camera" else DOUBLE))


def _hash_u8(p, c):
    """uint8 value of channel c of the source pixel at linear index p (int64, < 2^31)"""
    return ((p * _HASH_K[c]) >> 13) & 0xFF


def _fill_u8(torch, t):
    """t: (H, W, 3) uint8 CUDA tensor <- _hash_u8, in row chunks"""
    h, w, _ = t.shape
    step = max(1, (1 << 26) // w)
    for r0 in range(0, h, step):
        r1 = min(h, r0 + step)
        p = torch.arange(r0 * w, r1 * w, dtype=torch.int64, device="cuda")
        for c in range(3):
            t[r0:r1, :, c] = _hash_u8(p, c).to(torch.uint8).view(r1 - r0, w)
        del p


def _fill_index_f32(torch, t):
    """t: (H, W, 4) float32 CUDA tensor <- (p >> 16, p & 0xffff, 1, 1) (exact in float32)"""
    h, w, _ = t.shape
    step = max(1, (1 << 25) // w)
    t[..., 2:] = 1.0
    for r0 in range(0, h, step):
        r1 = min(h, r0 + step)
        p = torch.arange(r0 * w, r1 * w, dtype=torch.int64, device="cuda").view(r1 - r0, w)
        t[r0:r1, :, 0] = (p >> 16).to(torch.float32)
        t[r0:r1, :, 1] = (p & 0xFFFF).to(torch.float32)
        del p


def _want_u8(idx):
    """expected uint8 output of a hashed single-slot source for source indices idx (-1: black)"""
    p = np.maximum(idx, 0)
    out = np.stack([_hash_u8(p, c) for c in range(3)], axis=-1).astype(np.uint8)
    out[idx < 0] = 0
    return out


def _neighbours(idx, src_w):
    return [idx + s for s in (-1, 1, -src_w, src_w, -src_w - 1, -src_w + 1, src_w - 1, src_w + 1)]


def _check_u8(got, idx, src_w, what):
    """got (h, w, 3) uint8 against the hashed source's pixels at idx (h, w): equal, or an index flip
    on at most 1e-4 of the pixels"""
    want = _want_u8(idx)
    diff = (got != want).any(axis=2)
    n_diff = int(diff.sum())
    if n_diff == 0:
        return
    g, i = got[diff], idx[diff]
    explained = np.zeros(n_diff, bool)
    for n in _neighbours(i, src_w):
        explained |= (n >= 0) & (g == _want_u8(n)).all(axis=1)
    explained |= (i < 0) | ~g.any(axis=1)  # black / not black: the coordinate crossed the image border
    assert explained.all(), (what, int((~explained).sum()), n_diff)
    assert n_diff <= max(8, 1e-4 * diff.size), (what, n_diff)


def _check_index_f32(got, idx, src_w, what):
    """got (h, w, 4) float32 of an index-filled source: the index it carries against idx"""
    valid = got[..., 3] == 1.0
    assert np.all(valid | ~got.any(axis=2)), what  # a pixel is a whole source pixel or black
    carried = np.where(valid, got[..., 0].astype(np.int64) * 65536 + got[..., 1].astype(np.int64), -1)
    diff = carried != idx
    n_diff = int(diff.sum())
    if n_diff == 0:
        return
    c, i = carried[diff], idx[diff]
    explained = (c < 0) | (i < 0)
    for n in _neighbours(i, src_w):
        explained |= c == n
    assert explained.all(), (what, int((~explained).sum()), n_diff)
    assert n_diff <= max(8, 1e-4 * diff.size), (what, n_diff)


def _check_blend_band(got, frame, og, sg, rows, what):
    """rows (r0, r1) of an un-rotated output from a double-fisheye frame, with the acceptance of
    helpers.Oracle on that band -> 1-LSB blend pixels, pixels"""
    from oracle import c_port, numpy_port

    cmap = numpy_port.output_rays(og, rows=rows)
    blended = (c_port.source_index(og, (), sg, rows=rows) >= 0).all(axis=2)
    bad, px, degenerate, lsb = helpers.assert_like_oracle(got, frame, sg, cmap, what, blended=blended)
    return lsb, px


# ------------------------------------------------------------------------------------ plans and calls


class _Plan:
    def __init__(self, torch, og, rots, sg, channels=3):
        from photonbend_b200 import _native, engine

        self.torch, self.og, self.rots, self.sg = torch, og, rots, sg
        self.lib = _native.load()
        probe = torch.empty((1, 1, channels), dtype=torch.uint8, device="cuda").expand(sg["height"], sg["width"],
                                                                                      channels)
        geom = helpers.product_image(sg, probe)._source_geometry()
        self.desc = engine._remap_desc(helpers.product_map(og, rots).rays, geom, channels)
        self.handle = engine._plans.get(self.lib, self.desc, torch.cuda.current_device(), torch)

    def stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def _done(self, rc, ran, families, what):
        from photonbend_b200 import _native

        _native.check(rc)
        self.torch.cuda.synchronize()
        assert ran and set(ran) <= families, (what, ran)
        print(f"{what}: {ran}")

    def u8(self, src, s_stride, dst, d_stride, n, families, what):
        rc, ran = helpers.remap_launches(lambda: self.lib.pb_plan_remap_u8(
            self.handle, ctypes.c_void_p(src.data_ptr()), s_stride, ctypes.c_void_p(dst.data_ptr()), d_stride, n,
            self.stream()))
        self._done(rc, ran, families, what)

    def px(self, elem, src, s_stride, dst, d_stride, n, families, what):
        rc, ran = helpers.remap_launches(lambda: self.lib.pb_plan_remap_px(
            self.handle, elem, ctypes.c_void_p(src.data_ptr()), s_stride, ctypes.c_void_p(dst.data_ptr()), d_stride,
            n, self.stream()))
        if families is None:
            return rc, ran
        self._done(rc, ran, families, what)

    def frames(self, elem, rotations, src, s_stride, dst, d_stride, families, what):
        from oracle import numpy_port

        m = np.ascontiguousarray(np.stack([numpy_port.rotation_matrix(*r) for r in rotations]).reshape(-1, 9))
        rc, ran = helpers.remap_launches(lambda: self.lib.pb_plan_remap_frames_px(
            self.handle, elem, m.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ctypes.c_void_p(src.data_ptr()),
            s_stride, ctypes.c_void_p(dst.data_ptr()), d_stride, len(rotations), self.stream()))
        if families is None:
            return rc, ran
        self._done(rc, ran, families, what)

    def rows_u8(self, src, dst, r0, r1, families, what):
        rc, ran = helpers.remap_launches(lambda: self.lib.pb_plan_remap_rows_u8(
            self.handle, ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(dst.data_ptr()), r0, r1, self.stream()))
        self._done(rc, ran, families, what)


def _index(og, rots, sg, rows=None):
    from oracle import c_port

    return c_port.source_index(og, rots, sg, rows=rows)[..., 0]


def _report(what, **sizes):
    print(what + ": " + ", ".join(f"{k} {v / GIB:.2f} GiB" for k, v in sizes.items()))


# ------------------------------------------------------------------------------------ the 2^31 guard


@pytest.mark.parametrize("kind", ["equirect", "camera"])
def test_source_just_under_the_guard(torch_cuda, device_room, kind):
    """3 W H = 2^31 - 176: the last source size of the 32-bit offset kernels.  Single frames take
    direct / direct32 (rotated) or sep1 (a camera source, un-rotated), batches of 2 the tiled
    kernels; the output's last rows read the source's bottom rows, within 1 % of the 2^31-byte ceiling."""
    torch = torch_cuda
    sg = _geom(kind, GUARD_H, GUARD_W)
    P = 3 * GUARD_W * GUARD_H
    assert P < 1 << 31 and 3 * GUARD_W * (GUARD_H + 1) >= 1 << 31
    device_room(2 * P + (1 << 24), "two frames just under 2^31 bytes")
    _report(f"{kind} {GUARD_H}x{GUARD_W}", source=2 * P)
    src = torch.empty((2, GUARD_H, GUARD_W, 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, src[0])
    src[1].copy_(src[0])
    og = _geom("equirect", OUT_H, OUT_W)
    for rots in ((), ROT):
        plan = _Plan(torch, og, rots, sg)
        sep = kind == "camera" and not rots
        idx = _index(og, rots, sg)
        assert 3 * idx.max() >= 0.99 * (1 << 31), "the output reads within 1 % of the 2^31-byte ceiling"
        dst = torch.empty((2, OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda")
        one = {"sep1"} if sep else {"direct", "direct32"}
        plan.u8(src, P, dst, dst[0].numel(), 1, one, f"{kind} rots={len(rots)} x1")
        _check_u8(dst[0].cpu().numpy(), idx, GUARD_W, (kind, rots, 1))
        plan.u8(src, P, dst, dst[0].numel(), 2, {"tiled_sep"} if sep else {"tiled"}, f"{kind} rots={len(rots)} x2")
        got = dst.cpu().numpy()
        for k in range(2):
            _check_u8(got[k], idx, GUARD_W, (kind, rots, 2, k))
    del src, dst


@pytest.mark.parametrize("kind", ["equirect", "camera", "double"])
def test_source_just_over_the_guard(torch_cuda, device_room, kind):
    """One row more (3 W H >= 2^31): every call takes remap_generic_kernel, one frame and a batch of
    2 at source stride 0, and gives the oracle's pixels."""
    torch = torch_cuda
    h = GUARD_H + 1
    sg = _geom(kind, h, GUARD_W)
    P = 3 * GUARD_W * h
    device_room(P + (1 << 24), "a source just over 2^31 bytes")
    _report(f"{kind} {h}x{GUARD_W}", source=P)
    src = torch.empty((h, GUARD_W, 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, src)
    og = _geom("equirect", OUT_H, OUT_W)
    host = src.cpu().numpy() if kind == "double" else None
    for rots in ((), ROT):
        plan = _Plan(torch, og, rots, sg)
        dst = torch.empty((2, OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda")
        plan.u8(src, 0, dst, dst[0].numel(), 1, {"generic"}, f"{kind} rots={len(rots)} x1")
        single = dst[0].cpu().numpy()
        plan.u8(src, 0, dst, dst[0].numel(), 2, {"generic"}, f"{kind} rots={len(rots)} x2 stride 0")
        got = dst.cpu().numpy()
        assert np.array_equal(got[0], single) and np.array_equal(got[1], single), (kind, rots)
        if kind == "double":
            oracle = helpers.Oracle(og, rots, sg)
            oracle.check(single, host, (kind, rots))
            oracle.assert_lsb_share()
        else:
            _check_u8(single, _index(og, rots, sg), GUARD_W, (kind, rots))
    del src, dst, host


# ------------------------------------------------------------------------------------ the ABI maximum


@pytest.mark.parametrize("kind", ["equirect", "camera"])
def test_largest_source(torch_cuda, device_room, kind):
    """32767 x 65535 uint8 RGB (6.44 GB, past 2^32): the plan path (generic), the frames kernel's
    1-byte gather, and the explicit-map gather after a map edit (rows reversed)."""
    from photonbend_b200 import _native

    torch = torch_cuda
    h, w = 32767, 65535
    sg = _geom(kind, h, w)
    P = 3 * h * w
    device_room(P + (1 << 24), "the largest source")
    _report(f"{kind} {h}x{w}", source=P)
    src = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, src)
    og = _geom("equirect", OUT_H, OUT_W)
    plan = _Plan(torch, og, ROT, sg)
    idx = _index(og, ROT, sg)
    assert idx.max() >= (1 << 32) // 3, "the output reads past byte 2^32 of the source"
    dst = torch.empty((OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda")
    plan.u8(src, 0, dst, 0, 1, {"generic"}, f"{kind} plan")
    _check_u8(dst.cpu().numpy(), idx, w, (kind, "plan"))

    extra = ((0.05, -0.1, 0.2),)
    dst.fill_(0)
    plan.frames(1, extra, src, 0, dst, 0, {"frames"}, f"{kind} frames elem 1")
    _check_u8(dst.cpu().numpy(), _index(og, ROT + extra, sg), w, (kind, "frames"))

    cmap = torch.empty((OUT_H, OUT_W, 3), dtype=torch.float64, device="cuda")
    lib = _native.load()
    _native.check(lib.pb_materialize_map_f64(ctypes.byref(plan.desc), ctypes.c_void_p(cmap.data_ptr()), plan.stream()))
    cmap = cmap.flip(0).contiguous()  # the edit: the gather must follow the map, not the geometry
    dst.fill_(0)
    rc, ran = helpers.remap_launches(lambda: lib.pb_gather_from_map_u8(
        ctypes.byref(plan.desc.src), 3, ctypes.c_void_p(cmap.data_ptr()), OUT_H, OUT_W, ctypes.c_void_p(src.data_ptr()),
        ctypes.c_void_p(dst.data_ptr()), plan.stream()))
    plan._done(rc, ran, {"gather"}, f"{kind} gather after a map edit")
    _check_u8(dst.cpu().numpy(), idx[::-1], w, (kind, "gather"))
    del src, dst, cmap


def test_wide_source_past_4_gib(torch_cuda, device_room):
    """float32 RGBA camera source of 16384 x 32768 (8.6 GB): remap_wide_kernel separable and
    rotated, and the frames kernel."""
    torch = torch_cuda
    h, w = 16384, 32768
    sg = _geom("camera", h, w)
    P = 16 * h * w
    device_room(P + (1 << 24), "a float32 RGBA source past 4 GiB")
    _report(f"float32 RGBA camera {h}x{w}", source=P)
    src = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    _fill_index_f32(torch, src)
    og = _geom("equirect", OUT_H, OUT_W)
    dst = torch.empty((OUT_H, OUT_W, 4), dtype=torch.float32, device="cuda")
    for rots in ((), ROT):
        plan = _Plan(torch, og, rots, sg, channels=4)
        idx = _index(og, rots, sg)
        assert idx.max() >= (1 << 32) // 16, "the output reads past byte 2^32 of the source"
        dst.fill_(0)
        plan.px(4, src, 0, dst, 0, 1, {"wide"}, f"float32 rots={len(rots)}")
        _check_index_f32(dst.cpu().numpy(), idx, w, ("wide", rots))
        extra = ((0.1, 0.02, -0.3),)
        dst.fill_(0)
        plan.frames(4, extra, src, 0, dst, 0, {"frames"}, f"float32 frames rots={len(rots)}")
        _check_index_f32(dst.cpu().numpy(), _index(og, rots + extra, sg), w, ("frames", rots))
    del src, dst


# ------------------------------------------------------------------------------------ large outputs


def _bands(h, row_bytes):
    """first rows, the rows around byte offsets 2^31 and 2^32 (where the image has them), last rows"""
    bands = [(0, 64)]
    for edge in (1 << 31, 1 << 32):
        r = edge // row_bytes
        if r < h:
            bands.append((max(0, r - 40), min(h, r + 40)))
    bands.append((h - 64, h))
    return bands


def test_output_frame_past_2_gib(torch_cuda, device_room):
    """A 20480 x 40960 equirect output (2.5 GB) from a 3840 x 3840 camera source: sep1 un-rotated,
    direct32 rotated; row bands against the oracle."""
    torch = torch_cuda
    from photonbend_b200 import workloads

    sg = dict(workloads.WORKLOADS["T"]["src"])
    og = _geom("equirect", 20480, 40960)
    Q = 3 * og["height"] * og["width"]
    device_room(Q + (1 << 26), "an output frame past 2 GiB")
    _report("equirect 20480x40960 output", output=Q)
    src = torch.empty((sg["height"], sg["width"], 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, src)
    dst = torch.empty((og["height"], og["width"], 3), dtype=torch.uint8, device="cuda")
    for rots, families in (((), {"sep1"}), (ROT, {"direct32"})):
        plan = _Plan(torch, og, rots, sg)
        dst.fill_(0x5A)
        plan.u8(src, 0, dst, 0, 1, families, f"rots={len(rots)}")
        for r0, r1 in _bands(og["height"], 3 * og["width"]):
            _check_u8(dst[r0:r1].cpu().numpy(), _index(og, rots, sg, rows=(r0, r1)), sg["width"], (rots, r0))
    del src, dst


@pytest.mark.parametrize("workload", ["T", "cfg4"])
def test_batch_past_4_gib(torch_cuda, device_room, workload):
    """64 frames of the 8K target (tiled_sep) and of cfg4 (the box kernels) at source stride 0: 5.7 GB
    of output, frames 49 on past byte 2^32.  Frames on both sides of 2^32 and the last one equal the
    single-frame call, the last one the oracle on row bands.  A batch of two distinct frames checks
    that each output frame reads its own source frame."""
    torch = torch_cuda
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS[workload]
    og, sg = wl["out"], wl["src"]
    n = 64
    P, Q = 3 * sg["height"] * sg["width"], 3 * og["height"] * og["width"]
    assert 48 * Q < 1 << 32 < n * Q
    device_room(2 * P + (n + 1) * Q, f"{workload} x{n}")
    _report(f"{workload} x{n}", source=2 * P, output=n * Q)
    two = torch.empty((2, sg["height"], sg["width"], 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, two[0])
    two[1] = two[0].flip(1)
    dst = torch.empty((n, og["height"], og["width"], 3), dtype=torch.uint8, device="cuda")
    plan = _Plan(torch, og, (), sg)
    families = {"tiled_sep"} if sg["kind"] == "camera" else {"boxes1", "boxes2"}
    one = torch.empty((og["height"], og["width"], 3), dtype=torch.uint8, device="cuda")
    singles = []
    for k in range(2):
        plan.u8(two[k], P, one, Q, 1, {"sep1"}, f"{workload} single frame {k}")
        singles.append(one.cpu().numpy())
    plan.u8(two, P, dst, Q, 2, families, f"{workload} x2, two distinct frames")
    for k in range(2):
        assert np.array_equal(dst[k].cpu().numpy(), singles[k]), (workload, "x2", k)
    dst.fill_(CANARY)
    plan.u8(two[1], 0, dst, Q, n, families, f"{workload} x{n}, source stride 0")
    for k in (0, 47, 48, 49, 62, n - 1):
        assert np.array_equal(dst[k].cpu().numpy(), singles[1]), (workload, k)
    last = dst[n - 1].cpu().numpy()
    if sg["kind"] == "camera":
        for r0, r1 in _bands(og["height"], 3 * og["width"]):
            idx = _index(og, (), sg, rows=(r0, r1))
            # (frame 1 is frame 0 mirrored left to right)
            idx = np.where(idx >= 0, (idx // sg["width"]) * sg["width"] + sg["width"] - 1 - idx % sg["width"], -1)
            _check_u8(last[r0:r1], idx, sg["width"], (workload, r0))
    else:
        host = two[1].cpu().numpy()
        n_lsb = n_px = 0
        for r0, r1 in _bands(og["height"], 3 * og["width"]):
            lsb, px = _check_blend_band(last[r0:r1], host, og, sg, (r0, r1), (workload, r0))
            n_lsb, n_px = n_lsb + lsb, n_px + px
        assert n_lsb <= 2e-4 * n_px, (n_lsb, n_px)
    del two, dst, one


# ------------------------------------------------------------------------------------ row counts

TALL_W = 16  # 48-byte rows: 16-byte aligned, so the staged kernels take what they can


@pytest.mark.parametrize("height", [600_000, 65535 * 64 + 64])
def test_outputs_taller_than_a_grid(torch_cuda, device_room, height):
    """An equirect output of more than 65535 x 8 rows (the 2-D grids of the generic and the map
    kernels), and of more than 65535 x 64 (the wide and the frames kernels' tile rows), 16 columns
    wide.  Every entry point either gives the oracle's pixels on row bands, or refuses with
    PB_ERR_UNSUPPORTED and leaves the output as it was; which one is pinned here.  A rotated plan of
    the same output calibrates its FP32-first tier over every row."""
    from photonbend_b200 import _native

    torch = torch_cuda
    sg = {"kind": "camera", "height": 240, "width": 256, "lens": "equisolid", "fov": np.pi, "magnitude": 119.5}
    og = _geom("equirect", height, TALL_W)
    Q = 3 * height * TALL_W
    device_room(8 * Q + 24 * height * TALL_W, "a tall output")
    _report(f"equirect {height}x{TALL_W} output", output=Q)
    src = torch.empty((sg["height"], sg["width"], 3), dtype=torch.uint8, device="cuda")
    _fill_u8(torch, src)
    plan = _Plan(torch, og, (), sg)
    bands = [(0, 64), (height // 2 - 32, height // 2 + 32), (height - 100, height)]
    idx = {b: _index(og, (), sg, rows=b) for b in bands}
    tall = height > 65535 * 64

    def check(out, what):  # out: (height, TALL_W, 3) uint8 CUDA tensor
        for r0, r1 in bands:
            _check_u8(out[r0:r1].cpu().numpy(), idx[r0, r1], sg["width"], (what, r0))

    buf = torch.empty(2 * Q + 1, dtype=torch.uint8, device="cuda")
    dst = buf[:Q].view(height, TALL_W, 3)
    plan.u8(src, 0, dst, Q, 1, {"tiled_sep"} if tall else {"sep1"}, "u8 x1")
    check(dst, "u8 x1")
    odd = buf[1:].view(2, height, TALL_W, 3)  # a 1-byte offset: the generic kernel
    buf.fill_(CANARY)
    plan.u8(src, 0, odd, Q, 2, {"generic"}, "u8 x2 generic")
    check(odd[0], "generic frame 0")
    check(odd[1], "generic frame 1")

    band = torch.empty((height - 64, TALL_W, 3), dtype=torch.uint8, device="cuda")
    plan.rows_u8(src, band, 64, height, {"tiled_sep"}, "rows [64, H)")
    for r0, r1 in bands[1:]:
        _check_u8(band[r0 - 64:r1 - 64].cpu().numpy(), idx[r0, r1], sg["width"], ("rows", r0))
    del band

    # float32 RGB through remap_wide_kernel, uint8 through the frames kernel
    wsrc = src.to(torch.float32)
    wdst = torch.full((height, TALL_W, 3), -1.0, dtype=torch.float32, device="cuda")
    rc, ran = plan.px(4, wsrc, 0, wdst, 0, 1, None, "float32")
    torch.cuda.synchronize()
    if tall:
        assert rc == _native.PB_ERR_UNSUPPORTED and not ran, (rc, ran)
        assert b"65535 x 64" in plan.lib.pb_last_error()
        assert bool((wdst == -1.0).all())
    else:
        plan._done(rc, ran, {"wide"}, "float32")
        check(wdst.to(torch.uint8), "float32")
    del wsrc, wdst
    buf.fill_(CANARY)
    rc, ran = plan.frames(1, ((0.0, 0.0, 0.0),), src, 0, dst, 0, None, "frames")
    torch.cuda.synchronize()
    if tall:
        assert rc == _native.PB_ERR_UNSUPPORTED and not ran, (rc, ran)
        assert b"65535 x 64" in plan.lib.pb_last_error()
        assert bool((buf == CANARY).all())
    else:
        plan._done(rc, ran, {"frames"}, "frames")
        check(dst, "frames")

    # the coordinate map of every row, then the explicit-map gather
    lib = plan.lib
    cmap = torch.empty((height, TALL_W, 3), dtype=torch.float64, device="cuda")
    cmap.fill_(np.nan)
    rc, ran = helpers.remap_launches(lambda: lib.pb_materialize_map_f64(
        ctypes.byref(plan.desc), ctypes.c_void_p(cmap.data_ptr()), plan.stream()))
    plan._done(rc, ran, {"map"}, "materialize map")
    assert not bool(cmap.isnan().any())
    buf.fill_(CANARY)
    rc, ran = helpers.remap_launches(lambda: lib.pb_gather_from_map_u8(
        ctypes.byref(plan.desc.src), 3, ctypes.c_void_p(cmap.data_ptr()), height, TALL_W,
        ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(dst.data_ptr()), plan.stream()))
    plan._done(rc, ran, {"gather"}, "gather")
    check(dst, "gather")

    # a rotated plan: the FP32-first tier's calibration covers every row where the tier is on (pb_plan_create), the
    # diagnostic over every pixel returns, and one frame runs direct32 (the tiled kernel past
    # 65535 tile rows)
    rplan = _Plan(torch, og, ROT, sg)
    k = (ctypes.c_double * 2)()
    _native.check(lib.pb_debug_plan_fast32(rplan.handle, k))
    # (the tier is off for an output so tall that float rows lose precision: K = 0, nothing to calibrate)
    assert (k[0] > 0.0 and k[1] >= 0.0) or (k[0] == 0.0 and tall), tuple(k)
    stats = (ctypes.c_double * 6)()
    rc, ran = helpers.remap_launches(lambda: lib.pb_debug_fast32_stats(ctypes.byref(rplan.desc), stats, rplan.stream()))
    _native.check(rc)
    assert ran == {"diagnostic": 1} and stats[2] == height * TALL_W, (ran, tuple(stats))
    print(f"rotated plan: K {k[0]:.2f} from ratio {k[1]:.2f}; fast32 stats {tuple(stats)}")
    rplan.u8(src, 0, dst, 0, 1, {"tiled"} if tall else {"direct", "direct32"}, "rotated u8 x1")
    for r0, r1 in bands:
        _check_u8(dst[r0:r1].cpu().numpy(), _index(og, ROT, sg, rows=(r0, r1)), sg["width"], ("rotated", r0))
    del buf, dst, odd, cmap, src
