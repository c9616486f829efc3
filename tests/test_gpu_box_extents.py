"""Batches through a double-fisheye source stage each 16-row box of a tile's footprint at its own
first column and width (csrc/pb_boxes.cuh).  The plan's box table (pb_debug_plan_boxes) must cover
every source pixel a tile references and never be wider than the tile's bounding rectangle, and
the remapped bytes must equal those of the rectangle kernels (PB_BOX_EXTENTS=0)."""

import ctypes

import numpy as np
import pytest

import case_matrix
import helpers
from conftest import mismatch_report

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _geometries():
    from photonbend_b200 import workloads

    wl = workloads.WORKLOADS["cfg4"]  # cfg5 is the same geometry, 1024 frames
    cases = [("cfg4/cfg5", wl["out"], wl["src"])]
    rng = np.random.default_rng(2024)
    lenses = ("equidistant", "equisolid", "stereographic", "orthographic")
    for k in range(5):
        h = int(rng.integers(20, 90)) * 16
        fov = float(rng.uniform(180.0, 200.0))
        lens = lenses[k % len(lenses)]
        sg = {"kind": "double", "height": h, "width": 2 * h, "lens": lens, "fov": case_matrix.rad(fov)}
        oh = h + int(rng.integers(0, 4)) * 16
        og = {"kind": "equirect", "height": oh, "width": 2 * oh + int(rng.integers(0, 3)) * 32}
        cases.append((f"{lens} {fov:.2f} {h}", og, sg))
    return cases


GEOMETRIES = _geometries()


def _plan(torch, og, sg):
    from photonbend_b200 import _native, engine

    lib = _native.load()
    src = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
    desc = engine._remap_desc(helpers.product_map(og, ()).rays, src._source_geometry(), 3)
    return lib, engine._plans.get(lib, desc, torch.cuda.current_device(), torch)


def _box_table(torch, og, sg):
    from photonbend_b200 import _native

    lib, plan = _plan(torch, og, sg)
    dims = (ctypes.c_int32 * 3)()
    _native.check(lib.pb_debug_plan_boxes(plan, None, 0, dims))
    ty, tx, nb = dims
    assert (ty, tx, nb) == (-(-og["height"] // 64), -(-og["width"] // 32), 8), tuple(dims)
    table = np.zeros((ty, tx, 2, nb, 4), np.int32)
    _native.check(lib.pb_debug_plan_boxes(plan, table.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), table.size, dims))
    return table


def _stage_units(need):
    return np.maximum((need + 15) >> 4, 5) | 1


@pytest.mark.parametrize("name,og,sg", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_boxes_cover_the_footprint(torch_cuda, name, og, sg):
    from oracle import c_port

    table = _box_table(torch_cuda, og, sg)
    idx = c_port.source_index(og, (), sg)
    H, W, _ = idx.shape
    SW = sg["width"]
    ii, jj = np.mgrid[0:H, 0:W]
    ty, tx = ii // 64, jj // 32
    described = table[:, :, :, :, 1].min(axis=(2, 3)) >= 0
    assert described.mean() > 0.99, (name, described.mean())
    n_checked = 0
    for s in range(2):
        v = idx[..., s]
        m = (v >= 0) & described[ty, tx]
        y, x = v[m] // SW, v[m] % SW
        t = table[ty[m], tx[m], s]  # (n, boxes, 4)
        k = (y - t[:, 0, 3]) // 16
        assert k.min() >= 0 and k.max() < table.shape[3], name
        b = t[np.arange(k.size), k]
        assert np.all(b[:, 3] <= y) and np.all(y < b[:, 3] + 16), name
        assert np.all(b[:, 1] > 0), name
        assert np.all(b[:, 0] % 16 == 0), name
        assert np.all(b[:, 0] <= 3 * x) and np.all(3 * x + 3 <= b[:, 0] + 16 * b[:, 1]), name
        n_checked += k.size
        # no box is wider than the bounding rectangle of the tile's slot
        tile_id = (ty[m] * table.shape[1] + tx[m]).ravel()
        n_tiles = table.shape[0] * table.shape[1]
        xmin = np.full(n_tiles, np.iinfo(np.int64).max)
        xmax = np.full(n_tiles, -1)
        np.minimum.at(xmin, tile_id, x)
        np.maximum.at(xmax, tile_id, x)
        seen = xmax >= 0
        xb0 = (3 * xmin[seen]) & ~15
        rect_units = _stage_units(3 * xmax[seen] + 3 - xb0)
        units = table[:, :, s, :, 1].reshape(n_tiles, -1)[seen]
        assert np.all(units.max(axis=1) <= rect_units), name
        assert np.all(units.max(axis=1) % 2 == 1), name
    assert n_checked > 0


@pytest.mark.parametrize("name,og,sg", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_boxes_remap_like_rectangles(torch_cuda, name, og, sg, monkeypatch):
    torch = torch_cuda
    h, w = sg["height"], sg["width"]
    rng = np.random.default_rng(h)
    flat = [np.full((h, w, 3), v, np.uint8) for v in (200, 0, 255, 85, 170, 1)]
    noise = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(8)]
    ramp = (np.arange(h * w * 3, dtype=np.int64).reshape(h, w, 3) // 7 % 256).astype(np.uint8)
    frames = torch.from_numpy(np.stack(flat + noise + [ramp, case_matrix.case_image(sg, 77)])).cuda()
    assert frames.shape[0] == 16
    outs = {}
    for switch, families in (("1", {"boxes1", "boxes2"}), ("0", {"tiled_sep", "two_lens"})):
        monkeypatch.setenv("PB_BOX_EXTENTS", switch)
        outs[switch], ran = helpers.remap_launches(
            lambda: helpers.product_image(sg, frames).process_coordinate_map(helpers.product_map(og, ())).cpu().numpy())
        assert ran and set(ran) <= families, (switch, ran)  # the box kernels, and without them the rectangle kernels
    for k in range(16):
        assert np.array_equal(outs["1"][k], outs["0"][k]), (name, k, mismatch_report(outs["1"][k], outs["0"][k]))
    if h <= 800:  # and against the oracle, where that is quick
        from oracle import numpy_port

        for k in (0, 9, 14):
            want = numpy_port.remap(og, (), sg, frames[k].cpu().numpy())
            assert np.array_equal(outs["1"][k], want), (name, k)
