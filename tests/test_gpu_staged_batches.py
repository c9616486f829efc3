"""Batches through the TMA-staged kernels (remap_tiled_kernel in both modes, remap_boxes_kernel,
remap_wide_kernel for wider elements) on every image-kind pair, on frame counts around the ring of
kMaxGroups = 8 frames in flight, and on padded, misaligned and zero frame strides through the C ABI.

Every call reads the launch census (pb_debug_launch_counts) around it, so a test fails when the
routing sends it to another kernel than the one it is about.  The staged kernels must give the
bytes the generic kernel and the single-frame kernels give, and the NumPy oracle's pixels with the
acceptance of tests/test_gpu_parity.py::test_random_mid_size_geometries (helpers.Oracle)."""

import numpy as np
import pytest

import case_matrix
import helpers
import table_oracle

pytestmark = pytest.mark.gpu

rad = case_matrix.rad
LENSES = case_matrix.LENSES
CAMERA_FOV = {"equidistant": 200, "equisolid": 180, "orthographic": 170, "stereographic": 200, "rectilinear": 140,
              "thoby": 180}
DOUBLE_FOV = {"equidistant": 195, "equisolid": 190, "stereographic": 200, "thoby": 190}
ROTATION_SETS = ((), ((0.3, -0.2, 1.0),), ((rad(-90), 0.0, rad(195)), (0.1, 0.2, 0.3)))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


# ------------------------------------------------------------------------------------ geometries

# 16-byte aligned rows (3 channels, width % 16 == 0); output width = 16 (mod 32) and height not a
# multiple of 64: partial tiles on the right and bottom edges
OUT_H, OUT_W = 170, 336


def _out_geom(kind, lens):
    if kind == "equirect":
        return {"kind": "equirect", "height": OUT_H, "width": OUT_W}
    if kind == "camera":
        return {"kind": "camera", "height": OUT_H, "width": OUT_W, "lens": lens, "fov": rad(CAMERA_FOV[lens]),
                "magnitude": 150.5}
    lens = lens if lens in DOUBLE_FOV else "equidistant"
    return {"kind": "double", "height": OUT_H, "width": OUT_W, "lens": lens, "fov": rad(DOUBLE_FOV[lens])}


def _src_geom(kind, lens):
    if kind == "equirect":
        return {"kind": "equirect", "height": 192, "width": 384}
    if kind == "camera":
        return {"kind": "camera", "height": 240, "width": 256, "lens": lens, "fov": rad(CAMERA_FOV[lens]),
                "magnitude": 119.5}
    lens = lens if lens in DOUBLE_FOV else "equidistant"
    return {"kind": "double", "height": 192, "width": 384, "lens": lens, "fov": rad(DOUBLE_FOV[lens])}


def _staged_families(og, rots, sg):
    """The kernels plan_run routes an aligned batch to: the separable tables for an un-rotated
    panorama output of a lens source, generic rays (MODE 0) for everything else."""
    if og["kind"] == "equirect" and not rots and sg["kind"] == "camera":
        return {"tiled_sep"}
    if og["kind"] == "equirect" and not rots and sg["kind"] == "double":
        return {"boxes1", "boxes2"}  # one grid per tile class; a class may be empty
    return {"tiled"}


def _frames(sg, n, seed):
    """n distinct frames: flat ones (the double-fisheye blend on its truncation boundaries), noise,
    and shifted ramps."""
    h, w = sg["height"], sg["width"]
    rng = np.random.default_rng(seed)
    ramp = np.arange(h * w * 3, dtype=np.int64).reshape(h, w, 3) // 7
    flat = (200, 0, 255)
    out = []
    for k in range(n):
        if k % 3 == 0:
            j = k // 3
            out.append(np.full((h, w, 3), flat[j] if j < len(flat) else (200 + 37 * j) % 256, np.uint8))
        elif k % 3 == 1:
            out.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        else:
            out.append(((ramp + 11 * k) % 256).astype(np.uint8))
    return np.stack(out)


def _user_lens():
    """equisolid as a Lens of user callables: it runs through PB_LENS_TABLE"""
    from photonbend_b200.core.lens import Lens

    return Lens(lambda t: 2 * np.sin(t / 2), lambda r: 2 * np.arcsin(r / 2))


def _image(sg, array, user_lens=False):
    if user_lens:
        from photonbend_b200.core.projection import CameraImage

        return CameraImage(array, sg["fov"], _user_lens(), magnitude=sg.get("magnitude"))
    return helpers.product_image(sg, array)


def _remap(og, rots, sg, array, user_lens=False):
    """-> (output as numpy, {family: launches}) of one product call on a CUDA tensor"""
    cmap = helpers.product_map(og, rots)
    out, ran = helpers.remap_launches(lambda: _image(sg, array, user_lens).process_coordinate_map(cmap))
    return out.cpu().numpy(), ran


# ------------------------------------------------------------------------------------ B1: kind pairs


def _kind_pair_cases():
    """every (output, source) kind pair x ROTATION_SETS; the lenses of each (side, kind) go round
    all six (a double image maps rectilinear and orthographic to equidistant)"""
    cases = []
    drawn = {}

    def lens(side, kind):
        k = drawn[side, kind] = drawn.get((side, kind), -1) + 1
        return LENSES[(k + (side == "src")) % len(LENSES)]

    for ok in ("equirect", "camera", "double"):
        for sk in ("equirect", "camera", "double"):
            for r, rots in enumerate(ROTATION_SETS):
                user = ok == "equirect" and sk == "camera" and r == 0  # (the first camera source: equisolid)
                og, sg = _out_geom(ok, lens("out", ok)), _src_geom(sk, lens("src", sk))
                cid = f"{ok}-{og.get('lens', '')}<-{sk}-{sg.get('lens', '')}{'-user' if user else ''}-r{r}"
                cases.append(pytest.param(og, rots, sg, user, id=cid))
    return cases


@pytest.mark.parametrize("og,rots,sg,user_lens", _kind_pair_cases())
def test_kind_pair_batches(torch_cuda, og, rots, sg, user_lens):
    """9 distinct frames (one more than the ring holds) through the staged kernel the routing
    picks: the census names it, every frame matches the oracle, the batch equals the generic
    kernel's byte for byte (source at a 1-byte offset), frame 0 equals a single-frame call."""
    torch = torch_cuda
    frames = _frames(sg, 9, seed=sg["height"] + og["height"] + 7 * len(rots))
    dev = torch.from_numpy(frames).cuda()
    got, ran = _remap(og, rots, sg, dev, user_lens)
    staged = _staged_families(og, rots, sg)
    assert ran and set(ran) <= staged, (staged, ran)

    # a user lens: the table oracle of the tables the product built for this source
    with table_oracle.patched():
        oracle = helpers.Oracle(og, rots, table_oracle.geom_of(_image(sg, dev, True)) if user_lens else sg)
        for k in range(len(frames)):
            oracle.check(got[k], frames[k], k)
        oracle.assert_lsb_share()

    buf = torch.empty(dev.numel() + 1, dtype=torch.uint8, device="cuda")
    odd = buf[1:].view(dev.shape)
    odd.copy_(dev)
    generic, ran = _remap(og, rots, sg, odd, user_lens)
    assert ran == {"generic": 1}, ran
    for k in range(len(frames)):
        assert np.array_equal(got[k], generic[k]), (k, int((got[k] != generic[k]).any(axis=2).sum()))

    single, ran = _remap(og, rots, sg, dev[0], user_lens)
    assert ran and set(ran) <= {"direct", "direct32", "sep1"}, ran
    assert np.array_equal(single, got[0])


# ------------------------------------------------------------------------------------ B2: ring length

RING_FRAMES = (2, 3, 7, 8, 9, 16, 17, 40)
RING_PATHS = {
    "separable-camera": (_out_geom("equirect", None), (), _src_geom("camera", "equisolid")),
    "double-boxes": (_out_geom("equirect", None), (), _src_geom("double", "equidistant")),
    "camera-camera-rotated": (_out_geom("camera", "stereographic"), ROTATION_SETS[1], _src_geom("camera", "thoby")),
}


@pytest.mark.parametrize("path", list(RING_PATHS))
def test_frame_ring_lengths(torch_cuda, path, monkeypatch):
    """Batches of 2 .. 40 distinct frames: partial and several passes of the ring of frame groups
    (mbarrier parity flips every pass); every frame equals its single-frame call, and the single
    frames that end a batch match the oracle.  The double-fisheye path also runs with stage sizes so
    small that few groups fit (PB_ONE_BYTES, PB_REST_KIB are read on every call)."""
    torch = torch_cuda
    og, rots, sg = RING_PATHS[path]
    n_max = max(RING_FRAMES)
    frames = _frames(sg, n_max, seed=len(path))
    dev = torch.from_numpy(frames).cuda()
    singles = [_remap(og, rots, sg, dev[k])[0] for k in range(n_max)]
    oracle = helpers.Oracle(og, rots, sg)
    for k in sorted({0} | {n - 1 for n in RING_FRAMES}):
        oracle.check(singles[k], frames[k], (path, k))
    oracle.assert_lsb_share()
    staged = _staged_families(og, rots, sg)
    envs = [{}]
    if sg["kind"] == "double":
        envs.append({"PB_ONE_BYTES": "4096", "PB_REST_KIB": "8"})
    for env in envs:
        for name, value in env.items():
            monkeypatch.setenv(name, value)
        for n in RING_FRAMES:
            got, ran = _remap(og, rots, sg, dev[:n])
            assert ran and set(ran) <= staged, (env, n, ran)
            for k in range(n):
                assert np.array_equal(got[k], singles[k]), (env, n, k, int((got[k] != singles[k]).any(axis=2).sum()))
        for name in env:
            monkeypatch.delenv(name)


# ------------------------------------------------------------------------------------ B3: frame strides

CANARY = 0xA5
# (geometry, channels, element bytes); the 1-byte cases take pb_plan_remap_u8, the others pb_plan_remap_px
STRIDE_CASES = {
    "u8-separable-camera": (RING_PATHS["separable-camera"], 3, 1),
    "u8-double-boxes": (RING_PATHS["double-boxes"], 3, 1),
    "u8-camera-camera-rotated": (RING_PATHS["camera-camera-rotated"], 3, 1),
    "float32-separable-camera": (RING_PATHS["separable-camera"], 3, 4),
    "uint16-rgba-camera-rotated": (RING_PATHS["camera-camera-rotated"], 4, 2),
}


class _StridedPlan:
    """One plan called through the C ABI with explicit frame strides, always on the same pair of
    buffers (sized for the largest layout a test uses): the source's padding holds noise, the
    destination is filled with a canary before every call."""

    def __init__(self, torch, og, rots, sg, channels, elem, max_pad):
        from photonbend_b200 import _native, engine

        self.torch, self.elem = torch, elem
        self.lib = _native.load()
        src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], channels), np.uint8))
        desc = engine._remap_desc(helpers.product_map(og, rots).rays, src._source_geometry(), channels)
        self.plan = engine._plans.get(self.lib, desc, torch.cuda.current_device(), torch)
        self.P = sg["height"] * sg["width"] * channels * elem  # bytes of a packed source frame
        self.Q = og["height"] * og["width"] * channels * elem  # ... and of an output frame
        self.src = torch.empty(8 * (self.P + max_pad) + self.P, dtype=torch.uint8, device="cuda")
        self.dst = torch.empty(8 * (self.Q + max_pad) + self.Q + 64, dtype=torch.uint8, device="cuda")

    def run(self, frames, s_stride, d_stride):
        """frames (n, P) uint8 -> (outputs (n, Q), {family: launches}); checks the canary"""
        from photonbend_b200 import _native

        torch = self.torch
        n = len(frames)
        s_size = (n - 1) * s_stride + self.P
        d_size = (n - 1) * d_stride + self.Q + 64
        assert n <= 9 and self.src.numel() >= s_size and self.dst.numel() >= d_size
        host = np.random.default_rng(s_stride + n).integers(0, 256, self.src.numel(), dtype=np.uint8)
        for k in reversed(range(n)):  # (with a zero stride, frame 0 is the one left in place)
            host[k * s_stride:k * s_stride + self.P] = frames[k]
        self.src.copy_(torch.from_numpy(host))
        self.dst.fill_(CANARY)
        stream = torch.cuda.current_stream().cuda_stream

        def call():
            if self.elem == 1:
                return self.lib.pb_plan_remap_u8(self.plan, self.src.data_ptr(), s_stride, self.dst.data_ptr(), d_stride,
                                                 n, stream)
            return self.lib.pb_plan_remap_px(self.plan, self.elem, self.src.data_ptr(), s_stride, self.dst.data_ptr(),
                                             d_stride, n, stream)

        rc, ran = helpers.remap_launches(call)
        _native.check(rc)
        got = self.dst.cpu().numpy()
        written = np.zeros(got.size, bool)
        for k in range(n):
            written[k * d_stride:k * d_stride + self.Q] = True
        assert np.all(got[~written] == CANARY), (s_stride, d_stride, n, int((got[~written] != CANARY).sum()))
        return np.stack([got[k * d_stride:k * d_stride + self.Q] for k in range(n)]), ran


@pytest.mark.parametrize("case", list(STRIDE_CASES))
def test_frame_strides_and_map_caches(torch_cuda, case):
    """Frame k at src + k * src_frame_stride (include/pb_remap.h): (i) strides padded by 16-byte
    multiples stay on the staged kernel, (ii) padding that breaks 16-byte alignment takes the generic
    kernel, (iii) a zero source stride remaps one frame n times, (iv) one pair of buffers called with
    n = 2, 9, then 9 at larger strides must not reuse a tensor map encoded for another shape
    (cached_src_maps / cached_dst_map).  Nothing is written between output frames; every frame
    equals a single-frame call.  Wider elements take remap_wide_kernel, whose word width follows the
    strides (wide_vec)."""
    torch = torch_cuda
    (og, rots, sg), channels, elem = STRIDE_CASES[case]
    sp = _StridedPlan(torch, og, rots, sg, channels, elem, max_pad=80)
    P, Q = sp.P, sp.Q
    rng = np.random.default_rng(len(case))
    frames = rng.integers(0, 256, (9, P), dtype=np.uint8)
    frames[0] = 200  # a flat frame among the noise
    singles = [sp.run(frames[k:k + 1], P, Q)[0][0] for k in range(9)]
    staged = _staged_families(og, rots, sg) if elem == 1 else {"wide"}
    unaligned = {"generic"} if elem == 1 else {"wide"}

    def check(n, s_stride, d_stride, families, what=""):
        got, ran = sp.run(frames[:n], s_stride, d_stride)
        assert ran and set(ran) <= families, (what, ran)
        for k in range(n):
            want = singles[0] if s_stride == 0 else singles[k]
            assert np.array_equal(got[k], want), (what, k, int((got[k] != want).sum()))
        return ran

    check(9, P, Q, staged, what="packed")
    check(9, P + 48, Q + 80, staged, what="(i) padded by 16-byte multiples")
    check(9, P + 16, Q, staged, what="(i) source padded")
    # (wider elements: strides of whole elements that narrow the word width wide_vec picks)
    check(9, P + (elem if elem > 1 else 3), Q + 16, unaligned, what="(ii) source padding not 16-byte aligned")
    check(9, P, Q + (elem if elem > 1 else 8), unaligned, what="(ii) output padding not 16-byte aligned")
    # (iii): the staged kernels need a tensor map with a zero frame stride; without one the generic
    # kernel runs -- either way every output frame is frame 0's
    ran = check(9, 0, Q + 16, staged | unaligned, what="(iii) zero source stride")
    print(f"{case}: zero source stride ran {ran}")
    # (iv) the same buffers with another frame count, then larger strides (the tensor-map caches
    # are keyed by base, stride, frame count and width)
    check(2, P + 32, Q + 32, staged, what="(iv) n = 2")
    check(9, P + 32, Q + 32, staged, what="(iv) n = 9")
    check(9, P + 64, Q + 64, staged, what="(iv) n = 9, larger strides")
    check(3, P + 32, Q + 32, staged, what="(iv) n = 3 after the larger strides")


# ------------------------------------------------------------------------------------ B4: aligned fuzz


def _aligned_geometry(rng, role):
    """_random_geometry of tests/test_gpu_parity.py with every width a multiple of 16 (3-channel
    rows 16-byte aligned: batches take the staged kernels)."""
    kind = rng.choice(["equirect", "camera", "double"])
    if kind == "equirect":
        h = int(rng.integers(48, 260))
        return {"kind": "equirect", "height": h, "width": 16 * max(3, (2 * h + 8) // 16 + int(rng.choice([0, 0, 1])))}
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
        return {"kind": "double", "height": h, "width": 16 * max(4, (2 * h + 8) // 16 + int(rng.choice([0, 0, 1]))),
                "lens": lens, "fov": rad(float(rng.uniform(lo, hi)))}
    h, w = int(rng.integers(60, 420)), 16 * int(rng.integers(4, 27))
    if rng.random() < 0.5:
        w = 16 * max(4, (h + 8) // 16)
    mag = None if rng.random() < 0.4 else float(rng.uniform(0.4, 0.75) * min(h, w))
    return {"kind": "camera", "height": h, "width": w, "lens": lens, "fov": rad(float(rng.uniform(lo, hi))),
            "magnitude": mag}


def aligned_draws(fuzz_seed, n_draws=30):
    """[(og, rots, sg, n_frames)] of one seed"""
    rng = np.random.default_rng(fuzz_seed)
    draws = []
    for _ in range(n_draws):
        og, sg = _aligned_geometry(rng, "out"), _aligned_geometry(rng, "src")
        n_rot = int(rng.choice([0, 0, 1, 2]))
        rots = tuple(tuple(float(v) for v in rng.uniform(-3.2, 3.2, 3)) for _ in range(n_rot))
        draws.append((og, rots, sg, int(rng.choice([2, 3, 9]))))
    return draws


@pytest.mark.parametrize("fuzz_seed", [20261021, 11, 404])
def test_random_aligned_batches(torch_cuda, fuzz_seed):
    """Seeded fuzz of 16-aligned geometries with 2, 3 or 9 frames: every draw runs the staged kernel
    the routing predicts, with the acceptance of the unaligned fuzz; each seed reaches the tiled,
    the separable tiled and the box kernels."""
    torch = torch_cuda
    n_px = n_bad = n_degenerate = n_lsb = n_lsb_px = 0  # degenerate: draws
    seen = set()
    for case, (og, rots, sg, n_frames) in enumerate(aligned_draws(fuzz_seed)):
        frames = np.stack([case_matrix.case_image(sg, 9000 + 10 * case + k) for k in range(n_frames)])
        got, ran = _remap(og, rots, sg, torch.from_numpy(frames).cuda())
        cid = f"draw {case} {og} {rots} {sg} x{n_frames}"
        assert ran and set(ran) <= _staged_families(og, rots, sg), (cid, ran)
        seen |= set(ran)
        oracle = helpers.Oracle(og, rots, sg)
        degenerate = False
        for k in range(n_frames):
            bad, px, frame_degenerate = oracle.check(got[k], frames[k], (cid, k))
            n_bad += bad
            n_px += px
            degenerate |= frame_degenerate
        n_degenerate += degenerate
        n_lsb += oracle.n_lsb
        n_lsb_px += oracle.n_px
    print(f"aligned fuzz {fuzz_seed}: kernels {sorted(seen)}; {n_bad} differing pixels of {n_px} ({n_lsb} of the "
          f"1-LSB blend class); {n_degenerate} degenerate draws")
    assert n_lsb <= 2e-4 * n_lsb_px, (n_lsb, n_lsb_px)
    assert {"tiled", "tiled_sep"} <= seen and seen & {"boxes1", "boxes2"}, seen
    assert n_bad / n_px <= 1e-4, (n_bad, n_px)
    assert n_degenerate <= 6, n_degenerate
