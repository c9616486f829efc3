"""Cost per frame of a rotation per frame (pb_plan_remap_frames_px, csrc/pb_frames.cuh) against the two
ways a caller had before it, on cfg4 (the cfg5 video, stabilised), T and cfg2 with N = 16 frames and a
seeded wobble of a few degrees per frame on top of the workload's own rotations.  One JSON line per
(workload, route).

    python profiles/frame_rotation_bench.py [--out FILE] [--seconds 1.0]

Routes:
  A  one pb_plan_remap_frames_px call for the 16 frames (one launch: 16 <= 128 frames per launch);
  B  16 x remap_device(rays.rotated(M_k)) with fresh plans (the plan cache cleared first): what a
     per-frame rotation cost before, plan creation and its synchronisations included;
  C  16 single-frame launches through ONE cached plan with one fixed rotation: the resolve-bound
     floor of a calibrated FP32-first tier;
  C16  the same through a plan whose FP32-first tier keeps the un-calibrated K = 16 (PB_FP32_K=16
     while the plan is created), the bound route A uses: what of A's cost over C is that K.

Timing: A and C are captured as CUDA graphs of 20 calls that cycle over a pool of distinct source /
output buffers (together larger than 2 x the 126 MB L2) and replayed for at least ``--seconds``;
CUDA events around the window.  B has a host clock around 16 calls that end in a device
synchronise, repeated 5 times (median).  Compulsory bytes are the source frames read once plus the
output written.  ``mismatch_px``: pixels where A's frames differ from B's (must be 0).
"""

from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tests"), os.path.join(REPO, "profiles")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = ("cfg4", "T", "cfg2")
N = 16
WOBBLE_DEG = 3.0
L2_BYTES = 126 * 2**20
GRAPH_CALLS = 20


def graph_ms(torch, calls, seconds):
    """ms per call of ``calls`` (a list of GRAPH_CALLS thunks) captured as one CUDA graph."""
    for fn in calls[:3]:
        fn()
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        for fn in calls:
            fn()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    e1.synchronize()
    replays = max(3, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    e1.synchronize()
    window_ms = e0.elapsed_time(e1)
    del graph
    return window_ms / (replays * len(calls)), window_ms / 1e3


def run_workload(torch, name, seconds, peak):
    import helpers
    from photonbend_b200 import _native, engine, workloads
    from photonbend_b200.core.rotation import Rotation

    wl = workloads.WORKLOADS[name]
    sh, sw = wl["src"]["height"], wl["src"]["width"]
    oh, ow = workloads.output_shape(wl["out"])[:2]
    frame_bytes = sh * sw * 3 + oh * ow * 3
    call_bytes = N * frame_bytes
    pool = max(2, -(-2 * L2_BYTES // call_bytes))
    g = torch.Generator(device="cuda").manual_seed(1234)
    srcs = [torch.randint(0, 256, (N, sh, sw, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(pool)]
    outs = [torch.empty((N, oh, ow, 3), dtype=torch.uint8, device="cuda") for _ in range(pool)]
    rays = helpers.product_map(wl["out"], wl["rotations"]).rays
    geom = helpers.product_image(wl["src"], srcs[0][0])._source_geometry()
    import numpy as np

    rng = np.random.default_rng(5)
    w = math.radians(WOBBLE_DEG)
    mats = np.stack([Rotation(*rng.uniform(-w, w, 3)).rotation_matrix for _ in range(N)])
    lib = _native.load()
    base = {"workload": name, "frames": N, "wobble_deg": WOBBLE_DEG, "compulsory_bytes_per_frame": frame_bytes}
    rows = []

    def row(route, ms_frame, extra):
        gbs = frame_bytes / (ms_frame * 1e-3) / 1e9
        r = dict(base, route=route, us_per_frame=round(ms_frame * 1e3, 2), gbs=round(gbs, 1),
                 frac_of_peak=round(gbs / peak, 4))
        r.update(extra)
        rows.append(r)

    # A: one call per 16 frames (the first call creates the plan)
    engine.remap_frames_device(rays, geom, srcs[0], mats, outs[0])
    torch.cuda.synchronize()
    before = lib.pb_kernel_launches()
    engine.remap_frames_device(rays, geom, srcs[0], mats, outs[0])
    launches_a = lib.pb_kernel_launches() - before
    ms, window = graph_ms(torch, [lambda k=k: engine.remap_frames_device(rays, geom, srcs[k % pool], mats, outs[k % pool])
                                  for k in range(GRAPH_CALLS)], seconds)
    row("A: pb_plan_remap_frames_px, one call", ms / N,
        {"launches_per_call": launches_a, "window_s": round(window, 3),
         "l2": f"{pool} distinct source/output batches cycled ({pool * call_bytes / 1e6:.0f} MB)"})
    engine.remap_frames_device(rays, geom, srcs[0], mats, outs[0])
    torch.cuda.synchronize()
    got_a = outs[0].clone()

    # B: fresh plans, one per frame
    times = []
    for _ in range(5):
        engine.clear_plan_cache()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(N):
            engine.remap_device(rays.rotated(mats[k]), geom, srcs[0][k], outs[1][k])
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    engine.clear_plan_cache()
    mismatch = int((outs[1] != got_a).any(dim=-1).sum())
    row("B: 16 x remap_device with a fresh plan per frame", statistics.median(times) * 1e3 / N,
        {"host_clock_s": [round(t, 4) for t in times], "mismatch_px": mismatch})

    # C: 16 single-frame launches through one cached plan, one fixed rotation
    fixed = rays.rotated(mats[0])
    ms, window = graph_ms(torch, [lambda k=k: [engine.remap_device(fixed, geom, srcs[k % pool][f], outs[k % pool][f])
                                               for f in range(N)] for k in range(GRAPH_CALLS)], seconds)
    row("C: 16 single-frame launches, one cached plan", ms / N, {"window_s": round(window, 3)})

    # C16: as C through a plan created with the un-calibrated K = 16
    engine.clear_plan_cache()
    os.environ["PB_FP32_K"] = "16"
    try:
        engine.remap_device(fixed, geom, srcs[0][0], outs[0][0])  # the plan, created under K = 16
        torch.cuda.synchronize()
    finally:
        del os.environ["PB_FP32_K"]
    ms, window = graph_ms(torch, [lambda k=k: [engine.remap_device(fixed, geom, srcs[k % pool][f], outs[k % pool][f])
                                               for f in range(N)] for k in range(GRAPH_CALLS)], seconds)
    row("C16: as C, FP32-first tier at K = 16", ms / N, {"window_s": round(window, 3)})
    a, c = rows[0]["us_per_frame"], rows[2]["us_per_frame"]
    rows[0]["ratio_to_C"] = round(a / c, 3)
    rows[0]["ratio_to_B"] = round(a / rows[1]["us_per_frame"], 4)
    rows[0]["ratio_to_C16"] = round(a / rows[3]["us_per_frame"], 3)
    del srcs, outs
    engine.clear_plan_cache()
    torch.cuda.empty_cache()
    return rows


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--seconds", type=float, default=1.0, help="timed window per graph (>= 1 s)")
    args = ap.parse_args(argv)
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("frame_rotation_bench needs a CUDA device: nothing here is measured on the CPU")
    import bench
    from dtype_bench import card

    peak, peak_src = bench.measured_peak_gbs()
    name, watts = card(torch)
    lines = []
    for wl in WORKLOADS:
        for row in run_workload(torch, wl, max(1.0, args.seconds), peak):
            row.update({"card": name, "power_limit_w": watts, "peak_gbs": peak, "peak_source": peak_src})
            line = json.dumps(row)
            print(line, flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
