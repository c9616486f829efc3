"""The staged kernels at every footprint regime: source-to-output scales of 1/8 .. 8 and a source
4x taller than wide.

What runs inside remap_tiled_kernel and remap_boxes_kernel follows from the size of a tile's source
footprint, which follows from the scale: the lean ring of frame groups (and how many frames it keeps
in flight), the (frame, slot) item loop, or direct_tile for a footprint wider than the plan's widest
tensor map or larger than the stage area; a double-fisheye tile of more than 8 sixteen-row boxes is
handed to direct_tile as well.  An upscaled source stages minimum-width boxes that hang over its
bottom and right edges, where TMA fills with zeros.

A CPU model of the footprints, built from the C oracle's index map with the kernels' rules
(pb_tiled.cuh, pb_boxes.cuh) and the plan's staging sizes (pb_debug_plan_stage), sorts every tile
into these regimes.  The model must agree with the plan's box table (pb_debug_plan_boxes) on every
double-fisheye tile (check_box_table), and the sweep must reach every regime.  Every geometry then runs batches of 2
and 9 frames: the census names the kernel the routing predicts, every frame equals the generic
kernel's bytes and the NumPy oracle's pixels (helpers.Oracle), and frame 0 equals a single-frame
call (sep1, direct or direct32)."""

import ctypes

import numpy as np
import pytest

import helpers
from test_gpu_staged_batches import _frames, _staged_families

pytestmark = pytest.mark.gpu

OUT_H, OUT_W = 170, 336  # partial tiles on the right and bottom edges
SCALES = (1 / 8, 1 / 4, 1 / 2, 2, 4, 8)  # source pixels per output pixel along each axis
ROT = ((0.3, -0.2, 1.0),)
# pb_tiled.cuh / pb_boxes.cuh
TILE_H, TILE_W, BOX_ROWS, MAX_BOXES, MAX_GROUPS, MIN_UNITS = 64, 32, 16, 8, 8, 5
REGIMES = ("direct: too wide", "direct: too large", "direct: > 8 boxes", "item loop", "ring of 1", "ring of 2+",
           "min box at bottom-right")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


# ------------------------------------------------------------------------------------ geometries


def _w16(w):
    return 16 * max(1, int(round(w / 16)))  # 3-channel rows 16-byte aligned: batches stage


def _source(kind, scale, fov=195, tall=False):
    h = max(16, int(round(OUT_H * scale)))
    if kind == "camera":
        w = _w16(h / 4) if tall else _w16(OUT_W * scale)
        return {"kind": "camera", "height": h if not tall else 4 * w, "width": w, "lens": "equidistant",
                "fov": np.radians(200), "magnitude": None}
    if kind == "equirect":
        return {"kind": "equirect", "height": h, "width": _w16(2 * h)}
    return {"kind": "double", "height": h, "width": _w16(2 * h), "lens": "equidistant", "fov": np.radians(fov)}


def _geometries():
    og = {"kind": "equirect", "height": OUT_H, "width": OUT_W}
    cases = []
    for s in SCALES:
        tag = f"x{s:g}"
        cases.append((f"camera-{tag}", og, (), _source("camera", s)))
        for fov in (195, 181):
            cases.append((f"double{fov}-{tag}", og, (), _source("double", s, fov)))
        cases.append((f"rotated-camera-{tag}", og, ROT, _source("camera", s)))
        cases.append((f"rotated-equirect-{tag}", og, ROT, _source("equirect", s)))
        cases.append((f"rotated-double-{tag}", og, ROT, _source("double", s)))
    tall = _source("camera", 8, tall=True)  # 1360 x 336: 4x taller than wide
    cases.append(("tall-camera", og, (), tall))
    cases.append(("rotated-tall-camera", og, ROT, tall))
    return cases


GEOMETRIES = _geometries()


def _plan(torch, og, rots, sg):
    from photonbend_b200 import _native, engine

    lib = _native.load()
    src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
    desc = engine._remap_desc(helpers.product_map(og, rots).rays, src._source_geometry(), 3)
    return lib, engine._plans.get(lib, desc, torch.cuda.current_device(), torch)


def _stage(lib, plan):
    from photonbend_b200 import _native

    out = (ctypes.c_int32 * 8)()
    _native.check(lib.pb_debug_plan_stage(plan, out))
    keys = ("stage_bytes", "max_units", "n_buffers", "sep1_cap_camera", "sep1_cap", "sep1_cap_one", "boxes_one",
            "boxes_rest")
    return dict(zip(keys, out))


def _box_table(lib, plan):
    from photonbend_b200 import _native

    dims = (ctypes.c_int32 * 3)()
    _native.check(lib.pb_debug_plan_boxes(plan, None, 0, dims))
    ty, tx, nb = dims
    table = np.zeros((ty, tx, 2, nb, 4), np.int32)
    _native.check(lib.pb_debug_plan_boxes(plan, table.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), table.size, dims))
    return table


# ------------------------------------------------------------------------------------ the model


def stage_units(need):
    return np.maximum((need + 15) >> 4, MIN_UNITS) | 1


def footprints(og, rots, sg):
    """-> dict of (tiles_y, tiles_x, 2) arrays: by0, xb0, nbox, units, bytes (0 where a slot reads
    nothing), and (tiles_y, tiles_x) blended (a pixel reads both slots) and the (tiles_y,) tile rows
    whose every pixel row reads one slot only -- remap_tiled_kernel's footprint rules on the oracle's
    source index of every pixel (rows and columns past the image edge repeat the last one, which adds
    nothing to a footprint)"""
    from oracle import c_port

    idx = c_port.source_index(og, rots, sg)
    h, w = idx.shape[:2]
    ty, tx = -(-h // TILE_H), -(-w // TILE_W)
    pad = np.full((ty * TILE_H, tx * TILE_W, 2), -1, np.int64)
    pad[:h, :w] = idx
    t = pad.reshape(ty, TILE_H, tx, TILE_W, 2).transpose(0, 2, 4, 1, 3).reshape(ty, tx, 2, -1)
    sw = sg["width"]
    valid = t >= 0
    y, x = t // sw, t % sw
    big = np.int64(1) << 40
    min_y, max_y = np.where(valid, y, big).min(-1), np.where(valid, y, -1).max(-1)
    min_x, max_x = np.where(valid, x, big).min(-1), np.where(valid, x, -1).max(-1)
    any_px = max_y >= 0
    by0 = np.where(any_px, min_y, 0)
    xb0 = np.where(any_px, (min_x * 3) & ~15, 0)
    nbox = np.where(any_px, (max_y - by0 + BOX_ROWS) // BOX_ROWS, 0)
    units = np.where(any_px, stage_units(max_x * 3 + 3 - xb0), 0)
    both = (pad >= 0).all(axis=2)
    blended = both.reshape(ty, TILE_H, tx, TILE_W).any(axis=(1, 3))
    rows = np.concatenate([both[:h].any(axis=1), np.repeat(both[h - 1].any(), ty * TILE_H - h)])
    return {"by0": by0, "max_y": max_y, "xb0": xb0, "nbox": nbox, "units": units, "bytes": nbox * BOX_ROWS * 16 * units,
            "blended": blended, "unit_rows": ~rows.reshape(ty, TILE_H).any(axis=1)}


def classify_tiled(fp, st, n, dbl):
    """remap_tiled_kernel (pb_tiled.cuh, step 3): {regime: tiles} of a batch of n frames"""
    nslot = 2 if dbl else 1
    counts = {}
    for (ty, tx) in np.ndindex(fp["nbox"].shape[:2]):
        act = [s for s in range(nslot) if fp["nbox"][ty, tx, s] > 0]
        if not act:
            continue
        wide = any(fp["units"][ty, tx, s] > st["max_units"] for s in act)
        staged = not wide and all(fp["bytes"][ty, tx, s] <= st["stage_bytes"] for s in act)
        group = 128 + sum(int(fp["bytes"][ty, tx, s]) for s in act)
        n_groups = min(MAX_GROUPS, n, st["n_buffers"] * (st["stage_bytes"] + 128) // group)
        unit_weights = not (dbl and fp["blended"][ty, tx])
        lean = unit_weights and n_groups >= 1 and not wide
        if not staged and not lean:
            key = "direct: too wide" if wide else "direct: too large"
        elif lean:
            key = "ring of 1" if n_groups == 1 else "ring of 2+"
        else:
            key = "item loop"
        counts[key] = counts.get(key, 0) + 1
    return counts


def classify_boxes(fp, table, st, n):
    """remap_boxes_kernel (pb_boxes.cuh): {regime: tiles} of a batch of n frames.  A tile belongs to
    the one-lens class when one slot reads something and every row of its tile row sees one lens."""
    counts = {}
    for (ty, tx) in np.ndindex(fp["nbox"].shape[:2]):
        act = [s for s in range(2) if fp["nbox"][ty, tx, s] > 0]
        if not act:
            continue
        last = table[ty, tx, 1, MAX_BOXES - 1]
        one = len(act) == 1 and fp["unit_rows"][ty]
        ring = st["boxes_one"] if one else st["boxes_rest"]
        n_groups = min(MAX_GROUPS, n, (ring + 128) // (128 + int(last[2]) + BOX_ROWS * 16 * int(last[1])))
        if last[1] < 0:
            key = "direct: > 8 boxes"
        elif any(fp["units"][ty, tx, s] > st["max_units"] for s in act):
            key = "direct: too wide"
        elif n_groups < 1:
            key = "direct: too large"
        else:
            key = "ring of 1" if n_groups == 1 else "ring of 2+"
        counts[key] = counts.get(key, 0) + 1
    return counts


def edge_boxes(fp, sg):
    """(tile, slot) footprints of one minimum-width box that hangs over the source's bottom and right
    edges (the hardware zero-fills what lies outside)"""
    one = (fp["nbox"] == 1) & (fp["units"] == MIN_UNITS)
    return int((one & (fp["by0"] + BOX_ROWS > sg["height"]) & (fp["xb0"] + 16 * MIN_UNITS > 3 * sg["width"])).sum())


def check_box_table(fp, table, name):
    """the model against the plan's box table, every tile and slot: a tile the model needs more than
    8 boxes for is not described; described boxes cover the rows the model reads; and where the
    first rows agree, the box count of each slot is the model's.  -> slots whose first staged row lies above the model's: the plan's separable
    footprint bounds a tile's rows by the extreme lens radii of its rows, which may reach a few rows
    past the pixels the tile reads (more is staged than read, never less); such a tile may also need
    more than 8 boxes where the model needs 8 or fewer, and counts here too"""
    described = table[:, :, :, :, 1].min(axis=(2, 3)) >= 0
    fits = (fp["nbox"] <= MAX_BOXES).all(axis=2)
    assert not (described & ~fits).any(), (name, int((described & ~fits).sum()))
    staged = table[:, :, :, :, 1] > 0
    last = np.where(staged.any(axis=3), MAX_BOXES - 1 - np.argmax(staged[..., ::-1], axis=3), -1)
    m = described[..., None] & (fp["nbox"] > 0)
    first = table[..., 0, 3].astype(np.int64)
    assert np.all(first[m] <= fp["by0"][m]), (name, int((first[m] > fp["by0"][m]).sum()))
    assert np.all(fp["max_y"][m] < first[m] + BOX_ROWS * (last + 1)[m]), name
    same = m & (first == fp["by0"])  # the same first row: the same boxes
    assert np.array_equal((last + 1)[same], fp["nbox"][same]), (name, int(((last + 1)[same] != fp["nbox"][same]).sum()))
    assert not (described[..., None] & (fp["nbox"] == 0) & staged.any(axis=3)).any(), name
    return int((first[m] != fp["by0"][m]).sum()) + int((fits & ~described).sum())


def test_every_footprint_regime_is_reached(torch_cuda):
    """The model over the sweep, batches of 2 and 9 frames: every regime holds at least one tile, and
    the model agrees with every double-fisheye plan's box table."""
    torch = torch_cuda
    total = {k: 0 for k in REGIMES}
    sep1_global = shifted = 0
    for name, og, rots, sg in GEOMETRIES:
        lib, plan = _plan(torch, og, rots, sg)
        st = _stage(lib, plan)
        fp = footprints(og, rots, sg)
        dbl = sg["kind"] == "double"
        rows = []
        for n in (2, 9):
            if dbl and not rots:
                table = _box_table(lib, plan)
                if n == 2:
                    shifted += check_box_table(fp, table, name)
                counts = classify_boxes(fp, table, st, n)
            else:
                counts = classify_tiled(fp, st, n, dbl)
            rows.append(counts)
            for k, v in counts.items():
                total[k] += v
        edge = edge_boxes(fp, sg)
        total["min box at bottom-right"] += edge
        if sg["kind"] == "camera" and not rots:  # sep1: a footprint over its buffer gathers from global memory
            over = (fp["units"][..., 0] > 31) | (fp["bytes"][..., 0] > st["sep1_cap_camera"])
            sep1_global += int((over & (fp["nbox"][..., 0] > 0)).sum())
        print(f"{name}: src {sg['height']}x{sg['width']} stage {st['stage_bytes']} B, max_units {st['max_units']}, "
              f"x2 {rows[0]}, x9 {rows[1]}, edge boxes {edge}")
    print("tiles per regime over the sweep:", total, f"; single-frame camera tiles gathering from global memory "
          f"{sep1_global}; double-fisheye footprints the plan stages wider than the model {shifted}")
    missing = [k for k, v in total.items() if v == 0]
    assert not missing, (missing, total)


# ------------------------------------------------------------------------------------ the kernels


def _remap(og, rots, sg, array):
    cmap = helpers.product_map(og, rots)
    out, ran = helpers.remap_launches(lambda: helpers.product_image(sg, array).process_coordinate_map(cmap))
    return out.cpu().numpy(), ran


@pytest.mark.parametrize("name,og,rots,sg", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_scaled_batches(torch_cuda, name, og, rots, sg):
    """Batches of 2 and 9 frames: the staged kernel the routing predicts; every frame equals the
    generic kernel's bytes (source at a 1-byte offset) and the oracle; frame 0 equals a single-frame
    call; the batch of 2 is the first two frames of the batch of 9."""
    torch = torch_cuda
    frames = _frames(sg, 9, seed=sg["height"] * 7 + len(rots))
    dev = torch.from_numpy(frames).cuda()
    staged = _staged_families(og, rots, sg)
    got, ran = _remap(og, rots, sg, dev)
    assert ran and set(ran) <= staged, (name, staged, ran)
    two, ran = _remap(og, rots, sg, dev[:2])
    assert ran and set(ran) <= staged, (name, staged, ran)
    assert np.array_equal(two, got[:2]), name

    buf = torch.empty(dev.numel() + 1, dtype=torch.uint8, device="cuda")
    odd = buf[1:].view(dev.shape)
    odd.copy_(dev)
    generic, ran = _remap(og, rots, sg, odd)
    assert ran == {"generic": 1}, (name, ran)
    for k in range(9):
        assert np.array_equal(got[k], generic[k]), (name, k, int((got[k] != generic[k]).any(axis=2).sum()))

    single, ran = _remap(og, rots, sg, dev[0])
    one = {"sep1"} if staged <= {"tiled_sep", "boxes1", "boxes2"} else {"direct", "direct32"}
    assert ran and set(ran) <= one, (name, one, ran)
    assert np.array_equal(single, got[0]), name

    oracle = helpers.Oracle(og, rots, sg)
    for k in range(9):
        oracle.check(got[k], frames[k], (name, k))
    oracle.assert_lsb_share()


@pytest.mark.parametrize("scale", [1 / 8, 8])
def test_scaled_rows_wide_and_frame_rotations(torch_cuda, scale):
    """At the extreme scales, through the C ABI: a row band that starts on tile row 1 equals those rows
    of the single-frame call; float32 RGB through remap_wide_kernel gives the uint8 call's values; and
    pb_plan_remap_frames_px (uint8 and float32) equals the plan of the extended rotations."""
    from oracle import numpy_port
    from photonbend_b200 import _native

    torch = torch_cuda
    og = {"kind": "equirect", "height": OUT_H, "width": OUT_W}
    sg = _source("camera", scale)
    frame = torch.from_numpy(_frames(sg, 3, seed=5)[1]).cuda()  # noise
    lib, plan = _plan(torch, og, (), sg)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    Q = OUT_H * OUT_W * 3

    def call(fn, families, *args):
        rc, ran = helpers.remap_launches(lambda: fn(*args))
        _native.check(rc)
        torch.cuda.synchronize()
        assert ran and set(ran) <= families, (fn, ran)

    ptr = ctypes.c_void_p
    whole = torch.empty((OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda")
    call(lib.pb_plan_remap_u8, {"sep1"}, plan, ptr(frame.data_ptr()), 0, ptr(whole.data_ptr()), 0, 1, stream)
    band = torch.empty((OUT_H - 64, OUT_W, 3), dtype=torch.uint8, device="cuda")
    call(lib.pb_plan_remap_rows_u8, {"tiled_sep"}, plan, ptr(frame.data_ptr()), ptr(band.data_ptr()), 64, OUT_H, stream)
    assert torch.equal(band, whole[64:])

    wsrc = frame.to(torch.float32)
    wide = torch.empty((OUT_H, OUT_W, 3), dtype=torch.float32, device="cuda")
    call(lib.pb_plan_remap_px, {"wide"}, plan, 4, ptr(wsrc.data_ptr()), 0, ptr(wide.data_ptr()), 0, 1, stream)
    assert torch.equal(wide, whole.to(torch.float32))

    extra = (0.05, -0.1, 0.2)
    m = np.ascontiguousarray(numpy_port.rotation_matrix(*extra).reshape(1, 9))
    lib2, plan2 = _plan(torch, og, (extra,), sg)
    for elem, src, dtype in ((1, frame, torch.uint8), (4, wsrc, torch.float32)):
        want = torch.empty((OUT_H, OUT_W, 3), dtype=dtype, device="cuda")
        got = torch.empty_like(want)
        call(lib.pb_plan_remap_px, {"direct", "direct32"} if elem == 1 else {"wide"}, plan2, elem,
             ptr(src.data_ptr()), 0, ptr(want.data_ptr()), 0, 1, stream)
        call(lib.pb_plan_remap_frames_px, {"frames"}, plan, elem, m.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
             ptr(src.data_ptr()), 0, ptr(got.data_ptr()), Q * elem, 1, stream)
        assert torch.equal(got, want), (scale, elem, int((got != want).any(dim=2).sum()))
