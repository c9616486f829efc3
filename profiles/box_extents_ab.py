#!/usr/bin/env python
"""cfg5 x16 with the footprints staged box by box (PB_BOX_EXTENTS=1, csrc/pb_boxes.cuh) against
bounding rectangles issued by thread 0 (PB_BOX_EXTENTS=0), alternating in one process.

Each leg times the whole step and each tile class alone (PB_SKIP_CLASS=1: two-lens / blend-band grid
only, 2: one-lens grid only; the output of a one-class run is incomplete) with CUDA events around
`--iters` back-to-back calls of pb_plan_remap_u8 on 16-frame batches.  Two input batches alternate
(2 x 1.4 GB, far beyond the 126 MB of L2).  Also prints the bytes staged into shared memory per step,
from the plan's box table (pb_debug_plan_boxes) and from the bounding rectangles of the oracle's source
indices.  One JSON line per measurement.

    python profiles/box_extents_ab.py [--rounds 5] [--iters 20] [--frames 16]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


def staged_bytes(table, og, sg, frames):
    """bytes staged per step: (per-box extents, bounding rectangles), one-lens and two-lens tiles together"""
    from oracle import c_port

    boxes = int(np.maximum(table[..., 1], 0).astype(np.int64).sum()) * 16 * 16
    idx = c_port.source_index(og, (), sg)
    H, W, _ = idx.shape
    SW = sg["width"]
    ii, jj = np.mgrid[0:H, 0:W]
    tile = ((ii // 64) * table.shape[1] + jj // 32).ravel()
    n = table.shape[0] * table.shape[1]
    rect = 0
    for s in range(2):
        v = idx[..., s].ravel()
        m = v >= 0
        y, x, t = v[m] // SW, v[m] % SW, tile[m]
        lo = {k: np.full(n, np.iinfo(np.int64).max) for k in "xy"}
        hi = {k: np.full(n, -1) for k in "xy"}
        np.minimum.at(lo["x"], t, x)
        np.minimum.at(lo["y"], t, y)
        np.maximum.at(hi["x"], t, x)
        np.maximum.at(hi["y"], t, y)
        seen = hi["x"] >= 0
        xb0 = (3 * lo["x"][seen]) & ~15
        units = np.maximum((3 * hi["x"][seen] + 3 - xb0 + 15) >> 4, 5) | 1
        nbox = (hi["y"][seen] - lo["y"][seen] + 16) // 16
        rect += int((nbox * 16 * 16 * units).sum())
    return boxes * frames, rect * frames


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--frames", type=int, default=16)
    args = ap.parse_args()

    import torch

    import helpers
    from photonbend_b200 import _native, engine, workloads

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"what": "device", "name": torch.cuda.get_device_name(), "nvidia_smi": smi}), flush=True)
    wl = workloads.WORKLOADS["cfg5"]
    og, sg = wl["out"], wl["src"]
    lib = _native.load()
    src0 = helpers.product_image(sg, np.zeros((sg["height"], sg["width"], 3), np.uint8))
    desc = engine._remap_desc(helpers.product_map(og, ()).rays, src0._source_geometry(), 3)
    plan = engine._plans.get(lib, desc, torch.cuda.current_device(), torch)

    dims = (ctypes.c_int32 * 3)()
    _native.check(lib.pb_debug_plan_boxes(plan, None, 0, dims))
    table = np.zeros((dims[0], dims[1], 2, dims[2], 4), np.int32)
    _native.check(lib.pb_debug_plan_boxes(plan, table.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), table.size, dims))
    b, r = staged_bytes(table, og, sg, args.frames)
    print(json.dumps({"what": "staged_bytes_per_step", "workload": f"cfg5 x{args.frames}", "boxes": b, "rectangles": r,
                      "ratio": round(b / r, 4)}), flush=True)

    F, H, W = args.frames, sg["height"], sg["width"]
    gen = torch.Generator(device="cuda").manual_seed(5)
    srcs = [torch.randint(0, 256, (F, H, W, 3), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(2)]
    dst = torch.empty((F, og["height"], og["width"], 3), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def run(k):
        s = srcs[k & 1]
        _native.check(lib.pb_plan_remap_u8(plan, ctypes.c_void_p(s.data_ptr()), s[0].numel(), ctypes.c_void_p(dst.data_ptr()),
                                           dst[0].numel(), F, ctypes.c_void_p(stream)))

    def timed(boxed, skip):
        os.environ["PB_BOX_EXTENTS"] = "1" if boxed else "0"
        os.environ["PB_SKIP_CLASS"] = str(skip)
        for k in range(3):
            run(k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.iters):
            run(k)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.iters

    results = {}
    parts = {0: "step", 1: "two_lens_class", 2: "one_lens_class"}
    for rnd in range(args.rounds):
        for skip in (0, 1, 2):
            for boxed in ((False, True) if rnd % 2 == 0 else (True, False)):
                ms = timed(boxed, skip)
                key = (parts[skip], "boxes" if boxed else "rectangles")
                results.setdefault(key, []).append(ms)
                print(json.dumps({"what": "time", "round": rnd, "part": parts[skip], "staging": key[1], "ms": round(ms, 4)}),
                      flush=True)
    os.environ["PB_SKIP_CLASS"] = "0"
    for part in parts.values():
        r = results[(part, "rectangles")]
        bx = results[(part, "boxes")]
        print(json.dumps({"what": "summary", "part": part, "rectangles_median_ms": round(statistics.median(r), 4),
                          "boxes_median_ms": round(statistics.median(bx), 4),
                          "speedup": round(statistics.median(r) / statistics.median(bx), 4),
                          "boxes_faster_every_round": all(x < y for x, y in zip(bx, r))}), flush=True)


if __name__ == "__main__":
    main()
