"""Kernel time of a double-fisheye source blended in its own dtype (pb_blend.cuh,
DoubleCameraImage(..., keep_dtype=True)) next to the uint8 path, for uint16 RGB, float16 RGBA,
float32 RGB and float32 x 1, on cfg4 x1 (separable), cfg5 geometry x16 (separable) and cfg4 with
one rotation x1 (resolve_lookup per pixel).  One JSON line per (workload, dtype x C).

    python profiles/double_dtype_bench.py [--out FILE] [--seconds 1.0]

Timing as profiles/dtype_bench.py: every configuration is warmed up, then 20 launches that cycle
over a pool of distinct source / output buffers (together larger than 2 x the 126 MB L2) are
captured as one CUDA graph, replayed for at least ``--seconds``; CUDA events around the window.
Algorithmic bytes per frame: P x output pixels written + P x N_touched source pixels read once,
N_touched = the source pixels the un-rotated cfg4 geometry reads (tests/golden/full_configs.json;
the rotated row reuses it as the same order of magnitude).  ``mismatch_px``: pixels of frame 0 of
the last timed output, in the 512 rows around the blend band (ORACLE_ROWS), that differ from the
NumPy oracle (tests/typed_oracle.py: sample_double with the source dtype's cast) run on the device's
coordinate map; frames are uint8 noise widened to the dtype.  The card's name and power limit
are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tests"), os.path.join(REPO, "profiles")):
    if p not in sys.path:
        sys.path.insert(0, p)

MATRIX = [("cfg4", 1, ()), ("cfg5", 16, ()), ("cfg4", 1, ((0.3, -0.2, 1.0),))]
TYPES = [("uint8", 3), ("uint16", 3), ("float16", 4), ("float32", 3), ("float32", 1)]
L2_BYTES = 126 * 2**20
GRAPH_LAUNCHES = 20
ORACLE_ROWS = slice(1664, 2176)  # cfg4's blend band (sensor fov 195 degrees: rows 1760 .. 2080) and both sides


def n_touched():
    with open(os.path.join(REPO, "tests", "golden", "full_configs.json")) as fh:
        return int(json.load(fh)["cfg4"]["n_touched"])


def oracle_mismatch(torch, engine, sg, rays, frame, got):
    """Pixels of ``got`` (one output frame) that differ from the NumPy oracle on the device's map."""
    import numpy as np

    import typed_oracle

    name = str(frame.dtype).replace("torch.", "")
    cmap = engine.materialize_map_device(rays)[ORACLE_ROWS].cpu().numpy()
    with np.errstate(all="ignore"):
        want = typed_oracle.sample_double(sg, frame.cpu().numpy(), cmap, name)
    g = got[ORACLE_ROWS].cpu().numpy()
    same = (g == want) | (np.isnan(g) & np.isnan(want)) if g.dtype.kind == "f" else g == want
    return int((~same.reshape(g.shape[0], g.shape[1], -1).all(axis=2)).sum())


def run_one(torch, name, frames, rots, dtype_name, channels, seconds, peak, touched):
    import helpers
    from photonbend_b200 import _native, engine, workloads
    from photonbend_b200.core import lens as pb_lens
    from photonbend_b200.core.projection import DoubleCameraImage

    wl = workloads.WORKLOADS[name]
    sg = wl["src"]
    dtype = getattr(torch, dtype_name)
    e = torch.empty((), dtype=dtype).element_size()
    sh, sw = sg["height"], sg["width"]
    oh, ow = workloads.output_shape(wl["out"])[:2]
    src_bytes = frames * sh * sw * channels * e
    out_bytes = frames * oh * ow * channels * e
    pool = max(2, -(-2 * L2_BYTES // (src_bytes + out_bytes)))
    g = torch.Generator(device="cuda").manual_seed(1234)
    lead = (frames,) if frames > 1 else ()
    srcs = [torch.randint(0, 256, lead + (sh, sw, channels), dtype=torch.uint8, device="cuda", generator=g).to(dtype)
            for _ in range(pool)]
    outs = [torch.empty(lead + (oh, ow, channels), dtype=dtype, device="cuda") for _ in range(pool)]
    rays = helpers.product_map(wl["out"], rots).rays
    image = srcs[0][0] if frames > 1 else srcs[0]
    geom = DoubleCameraImage(image, sg["fov"], getattr(pb_lens, sg["lens"])(), keep_dtype=True)._source_geometry()

    for k in range(3):  # plan, module load
        engine.remap_device(rays, geom, srcs[k % pool], outs[k % pool])
    torch.cuda.synchronize()
    before = _native.launch_counts()
    engine.remap_device(rays, geom, srcs[0], outs[0])
    after = _native.launch_counts()
    launches = {k: after[k] - before[k] for k in after if after[k] != before[k]}
    torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        for k in range(GRAPH_LAUNCHES):
            engine.remap_device(rays, geom, srcs[k % pool], outs[k % pool])
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
    us = window_ms * 1e3 / (replays * GRAPH_LAUNCHES)

    last = (GRAPH_LAUNCHES - 1) % pool
    first = (lambda t: t[0]) if frames > 1 else (lambda t: t)
    mismatch = oracle_mismatch(torch, engine, sg, rays, first(srcs[last]), first(outs[last]))
    algo = frames * channels * e * (oh * ow + touched)
    gbs = algo / (us * 1e-6) / 1e9
    row = {"workload": name, "frames": frames, "rotations": len(rots), "dtype": dtype_name, "channels": channels,
           "px_bytes": channels * e,
           "path": "uint8 kernels" if dtype_name == "uint8" else "typed blend (remap_blend_kernel)",
           "launches_per_call": launches, "us_per_launch": round(us, 2), "window_s": round(window_ms / 1e3, 3),
           "algorithmic_bytes": algo, "gbs": round(gbs, 1), "frac_of_peak": round(gbs / peak, 4),
           "l2": f"{pool} distinct source/output buffers cycled ({pool * (src_bytes + out_bytes) / 1e6:.0f} MB)",
           "mismatch_px": mismatch}
    del graph, srcs, outs
    torch.cuda.empty_cache()
    return row


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--seconds", type=float, default=1.0, help="timed window per configuration (>= 1 s)")
    args = ap.parse_args(argv)
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("double_dtype_bench needs a CUDA device: nothing here is measured on the CPU")
    import bench
    from dtype_bench import card

    peak, peak_src = bench.measured_peak_gbs()
    name, watts = card(torch)
    touched = n_touched()
    rows = []
    for wl, frames, rots in MATRIX:
        base_us = None
        for dtype_name, channels in TYPES:
            row = run_one(torch, wl, frames, rots, dtype_name, channels, max(1.0, args.seconds), peak, touched)
            if dtype_name == "uint8":
                base_us = row["us_per_launch"]
            else:
                row["ratio_to_uint8_rgb"] = round(row["us_per_launch"] / base_us, 3)
            row.update({"card": name, "power_limit_w": watts, "peak_gbs": peak, "peak_source": peak_src})
            line = json.dumps(row)
            print(line, flush=True)
            rows.append(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
