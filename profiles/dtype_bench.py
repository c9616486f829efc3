"""Kernel time of the remap by element type: the uint8 path next to the wide kernel (pb_wide.cuh)
for uint16 RGB, float16 RGBA, float32 RGB and float32 x 1 (a depth map), on T x1, T x8, cfg2 x1
and cfg3 x1.  One JSON line per (workload, dtype x C, frames).

    python profiles/dtype_bench.py [--out FILE] [--seconds 1.0]

Timing: every configuration is warmed up, then 20 launches that cycle over a pool of distinct
source / output buffers (together larger than the 126 MB L2) are captured as one CUDA graph and
the graph is replayed for at least ``--seconds``; CUDA events around the whole window give the
time per launch (events around single launches would also time the host's way to the launch).
Compulsory bytes are the source read once plus the output written, from the shapes.  Afterwards
the wide output of the last launch is checked against the uint8 path run on its bytes in groups
of <= 4 bytes (``mismatch_px``).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

MATRIX = [("T", 1), ("T", 8), ("cfg2", 1), ("cfg3", 1)]
TYPES = [("uint8", 3), ("uint16", 3), ("float16", 4), ("float32", 3), ("float32", 1)]
L2_BYTES = 126 * 2**20
GRAPH_LAUNCHES = 20


def card(torch):
    """(name, power limit in W or None) of the current device, read now."""
    name = torch.cuda.get_device_name()
    try:
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        return name, nv.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        return name, float(out.stdout.strip().splitlines()[0])
    except Exception:
        return name, None


def byte_group_mismatch(torch, engine, rays, geom, src, got):
    """Pixels where ``got`` differs from the uint8 path run on the bytes of ``src``, <= 4 at a time."""
    b = src.view(torch.uint8)
    want = torch.cat([engine.remap_device(rays, geom, b[..., k:k + 4].contiguous()) for k in range(0, b.shape[-1], 4)],
                     dim=-1)
    return int((got.view(torch.uint8) != want).reshape(-1, want.shape[-1]).any(dim=1).sum())


def run_one(torch, name, frames, dtype_name, channels, seconds, peak):
    import helpers
    from photonbend_b200 import _native, engine, workloads

    wl = workloads.WORKLOADS[name]
    dtype = getattr(torch, dtype_name)
    e = torch.empty((), dtype=dtype).element_size()
    sh, sw = wl["src"]["height"], wl["src"]["width"]
    oh, ow = workloads.output_shape(wl["out"])[:2]
    src_bytes = frames * sh * sw * channels * e
    out_bytes = frames * oh * ow * channels * e
    pool = max(2, -(-2 * L2_BYTES // (src_bytes + out_bytes)))  # buffers of a cycle: > 2x L2 together
    g = torch.Generator(device="cuda").manual_seed(1234)
    lead = (frames,) if frames > 1 else ()
    srcs = [torch.randint(0, 256, lead + (sh, sw, channels * e), dtype=torch.uint8, device="cuda", generator=g)
            .view(dtype) for _ in range(pool)]
    outs = [torch.empty(lead + (oh, ow, channels), dtype=dtype, device="cuda") for _ in range(pool)]
    rays = helpers.product_map(wl["out"], wl["rotations"]).rays
    geom = helpers.product_image(wl["src"], srcs[0][0] if frames > 1 else srcs[0])._source_geometry()

    lib = _native.load()
    for k in range(3):  # plan, kernel attributes, module load
        engine.remap_device(rays, geom, srcs[k % pool], outs[k % pool])
    torch.cuda.synchronize()
    before = lib.pb_kernel_launches()
    engine.remap_device(rays, geom, srcs[0], outs[0])
    launches = lib.pb_kernel_launches() - before
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
    ms = window_ms / (replays * GRAPH_LAUNCHES)

    last = (GRAPH_LAUNCHES - 1) % pool
    mismatch = None
    if e > 1:
        mismatch = byte_group_mismatch(torch, engine, rays, geom, srcs[last], outs[last])
    gbs = (src_bytes + out_bytes) / (ms * 1e-3) / 1e9
    row = {"workload": name, "frames": frames, "dtype": dtype_name, "channels": channels, "px_bytes": channels * e,
           "path": "uint8 (pb_plan_remap_u8)" if e == 1 else "wide (pb_plan_remap_px, remap_wide_kernel)",
           "ms_per_launch": round(ms, 5), "window_s": round(window_ms / 1e3, 3),
           "launches_per_call": launches, "compulsory_bytes": src_bytes + out_bytes,
           "gbs": round(gbs, 1), "frac_of_peak": round(gbs / peak, 4),
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
        raise SystemExit("dtype_bench needs a CUDA device: nothing here is measured on the CPU")
    import bench

    peak, peak_src = bench.measured_peak_gbs()
    name, watts = card(torch)
    rows = []
    for wl, frames in MATRIX:
        base_ms = None
        for dtype_name, channels in TYPES:
            row = run_one(torch, wl, frames, dtype_name, channels, max(1.0, args.seconds), peak)
            if dtype_name == "uint8":
                base_ms = row["ms_per_launch"]
            else:
                row["ratio_to_uint8_rgb"] = round(row["ms_per_launch"] / base_ms, 3)
            row.update({"card": name, "power_limit_w": watts, "peak_gbs": peak, "peak_source": peak_src})
            line = json.dumps(row)
            print(line, flush=True)
            rows.append(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
