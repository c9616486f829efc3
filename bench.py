#!/usr/bin/env python
"""bench.py -- throughput of the remap path on B200 (and of the reference's CPU path beside it).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg5|T|cfg1..cfg4]
    python bench.py --impl reference [...]          # the reference's CPU algorithm, host cores
    python bench.py --dump-outputs DIR [...]        # also write the last timed step's output to DIR/*.npy
    torchrun ... bench.py --gpus N ...              # one rank per GPU (driver launches this)

One JSON line on stdout (rank 0).  Metric: output Gpix/s, whole job.  ``value`` is timed over
exactly --steps steps (a burst of milliseconds); ``sustained`` repeats the same steps for >= 1.5 s
with its own clock record; ``parity`` compares frames of both timed paths with the CPU oracle.

A "step" is one pass of the hot path over one batch of ``--frames`` synthetic frames that share
the workload's geometry: ONE pb_remap_u8 launch (the source index of an output pixel is resolved
once and applied to every frame of the batch).  Inputs are resident in HBM before the timed
region; every step touches frames*(src+dst) bytes >> the 126 MB L2, so no L2 flush is needed.
With N ranks every rank owns its own batch (frames sharded k mod N, no collective): weak scaling.

``e2e`` is the same metric through the public API (photonbend_b200.batch.FramePipeline) with
pinned HOST buffers: every frame's H2D copy and D2H copy are inside the timed region.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from photonbend_b200 import workloads  # noqa: E402

METRIC = "output_gpix_per_s"
UNIT = "Gpix/s"
CHANNELS = 3


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------
# accounting


def golden_info(name: str) -> dict:
    key = "cfg4" if name == "cfg5" else name
    with open(os.path.join(REPO, "tests", "golden", "full_configs.json")) as fh:
        return json.load(fh)[key]


def algorithmic_bytes_per_frame(name: str) -> int:
    """B_alg = C*Ho*Wo (every output byte written once) + C*N_touched (every referenced source
    pixel read once); N_touched counted by the oracle (tests/golden/full_configs.json)."""
    info = golden_info(name)
    return CHANNELS * (info["out_pixels"] + info["n_touched"])


def committed_traffic(name: str, frames: int):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/)."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        entry = json.load(fh).get(f"{name}:{frames}")
    return entry["bytes"] if entry else None


def committed_counters(name: str, frames: int):
    """Issue-side counters of the same capture (instructions per output pixel, FP64 pipe, issue slots)."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        entry = json.load(fh).get(f"{name}:{frames}") or {}
    keys = ("inst_per_px", "fp64_pipe_pct", "issue_active_pct", "source")
    return {k: entry[k] for k in keys if k in entry} or None


def bench_config(name: str, frames: int) -> dict:
    """The workload both arms (--impl b200 / reference) are quoted on."""
    wl = workloads.WORKLOADS[name]
    info = golden_info(name)
    return {"workload": name, "title": wl["title"], "frames_per_step_per_gpu": frames,
            "out": f"{info['shape'][1]}x{info['shape'][0]}x{CHANNELS} u8",
            "l2": "inputs larger than L2: each step reads and writes "
                  f"{frames} distinct frames ({frames * (info['src_pixels'] + info['out_pixels']) * 3 / 1e6:.0f} MB)",
            "sharding": "frames k mod N per GPU, no collective"}


def measured_peak_gbs():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores.
#
# kind "reference": the UNMODIFIED reference package, copied by __graft_entry__.build() to the
# git-ignored oracle/_ref/ (it is pure Python + NumPy and imports as it lies), driven through its
# own three-call protocol
# (photonbend/core/__init__.py:66-92).  The reference is single-threaded; to use every host core
# the coordinate map is cut into row bands, one worker process per band (the protocol takes any
# (h, w, 3) slice of a map, bit-identically -- checked below against the golden hash).
# kind "port": oracle/numpy_port.py, the stated fallback when oracle/_ref is absent.

REF_DIR = os.path.join(REPO, "oracle", "_ref")


def live_reference():
    """The reference's modules from oracle/_ref, or None."""
    if not os.path.isdir(os.path.join(REF_DIR, "photonbend", "core")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import warnings

    warnings.simplefilter("ignore")  # benign NumPy RuntimeWarnings of the reference
    from photonbend.core import lens, projection, rotation

    return {"lens": lens, "projection": projection, "rotation": rotation}


def _ref_object(ref, geom, array):
    pj = ref["projection"]
    if geom["kind"] == "equirect":
        return pj.PanoramaImage(array)
    lens = getattr(ref["lens"], geom["lens"])()
    if geom["kind"] == "camera":
        return pj.CameraImage(array, geom["fov"], lens, magnitude=geom.get("magnitude"))
    return pj.DoubleCameraImage(array, geom["fov"], lens)


_CPU = {}  # state inherited by forked workers: image, reference objects, coordinate map


def _live_band_worker(args):
    r0, r1 = args
    ref, wl = _CPU["ref"], _CPU["wl"]
    band = _CPU["cmap"][r0:r1]
    for pyr in wl["rotations"]:
        band = ref["rotation"].Rotation(*pyr).rotate_coordinate_map(band)
    _CPU["out"][r0:r1] = _CPU["src"].process_coordinate_map(band)  # shared memory: nothing is pickled
    return r0, r1


def _port_band_worker(args):
    r0, r1 = args
    from oracle import numpy_port

    wl = _CPU["wl"]
    _CPU["out"][r0:r1] = numpy_port.remap(wl["out"], wl["rotations"], wl["src"], _CPU["image"], rows=(r0, r1))
    return r0, r1


class CpuArm:
    """One workload on all host cores; ``step(band_rows)`` remaps ``procs`` row bands of
    ``band_rows`` rows spread evenly over one frame (the whole frame when band_rows = H / procs)."""

    def __init__(self, name: str):
        import multiprocessing as mp

        os.environ.setdefault("OMP_NUM_THREADS", "1")
        self.name = name
        self.wl = workloads.WORKLOADS[name]
        self.procs = len(os.sched_getaffinity(0))
        self.h = self.wl["out"]["height"]
        self.w = workloads.output_shape(self.wl["out"])[1]
        self.ctx = mp.get_context("fork")
        self.ref = live_reference()
        self.kind = "reference" if self.ref else "port"
        self.stream = "frames" in self.wl  # a video: one geometry, many frames
        image = workloads.source_image(self.wl)
        _CPU.update(wl=self.wl, image=image, ref=self.ref)
        if self.ref:
            _CPU["src"] = _ref_object(self.ref, self.wl["src"], image)
            self.dst = _ref_object(self.ref, self.wl["out"],
                                   np.zeros((self.h, self.wl["out"]["width"], 3), np.uint8))
            if self.stream:
                # the geometry of a stream is fixed: its coordinate map is built once and serves
                # every frame (0.5 s of the reference's 9.5 s per frame; left out of the steps)
                _CPU["cmap"] = self.dst.get_coordinate_map()
        self.full_band = -(-self.h // self.procs)
        # the workers write their rows into one shared output frame
        shared = self.ctx.RawArray("B", self.h * self.w * CHANNELS)
        _CPU["out"] = np.frombuffer(shared, dtype=np.uint8).reshape(self.h, self.w, CHANNELS)

    def step(self, band_rows: int):
        """-> (pixels, seconds, rows covered); the rows land in the shared output frame"""
        band_rows = max(1, min(band_rows, self.full_band))
        bands = []
        for k in range(self.procs):
            r0 = min(k * self.full_band, self.h)
            r1 = min(r0 + band_rows, self.h)
            if r1 > r0:
                bands.append((r0, r1))
        t0 = time.perf_counter()
        if self.ref and not self.stream:
            _CPU["cmap"] = self.dst.get_coordinate_map()  # a single image: the map is part of the call
        with self.ctx.Pool(self.procs) as pool:
            res = pool.map(_live_band_worker if self.ref else _port_band_worker, bands, chunksize=1)
        dt = time.perf_counter() - t0
        rows = sum(r1 - r0 for r0, r1 in res)
        return rows * self.w, dt, rows

    def pick_band_rows(self, seconds_per_step: float) -> int:
        px, dt, _ = self.step(16)
        rows = int(16 * seconds_per_step / max(dt, 1e-3))
        return max(16, min(self.full_band, rows))

    def whole_frame_matches_golden(self, rows: int):
        """sha256 of a full-frame step against the reference output hash committed in tests/golden."""
        import hashlib

        if rows != self.h:
            return None
        return hashlib.sha256(_CPU["out"].tobytes()).hexdigest() == golden_info(self.name)["out_sha256"]

    def describe(self, band_rows, px, dt, steps=1):
        what = ("the unmodified reference (oracle/_ref/photonbend, three-call protocol"
                + ("; coordinate map of the stream built once, outside the steps)" if self.stream else ")")
                if self.ref else "oracle/numpy_port.py (NumPy restatement, bit-identical to the reference; oracle/_ref absent)")
        frac = band_rows * self.procs / self.h
        return (f"{what}, {self.procs} worker processes, one row band of {band_rows} rows each per step "
                f"({min(1.0, frac):.2f} of a {self.h}-row {self.name} frame), {dt / steps:.2f} s wall per step")


def cpu_baseline(name: str, budget_s: float = 20.0):
    arm = CpuArm(name)
    rows = arm.pick_band_rows(budget_s / 3)
    tot_px, tot_dt, n, match = 0, 0.0, 0, None
    while n < 3 and (tot_dt < budget_s * 0.7 or n == 0):
        px, dt, out = arm.step(rows)
        tot_px += px
        tot_dt += dt
        n += 1
        if match is None:
            match = arm.whole_frame_matches_golden(out)
    res = {"value": tot_px / tot_dt / 1e9, "unit": UNIT, "cores": arm.procs, "kind": arm.kind,
           "sample": arm.describe(rows, tot_px, tot_dt, n) + f", {n} steps"}
    if match is not None:
        res["output_sha256_matches_reference_golden"] = bool(match)
    return res


def c_port_rate(name: str):
    """Scalar C port of the same algorithm on all cores, for context (not the reference arm)."""
    from oracle import c_port

    wl = workloads.WORKLOADS[name]
    image = workloads.source_image(wl)
    h = wl["out"]["height"]
    rows = (0, h)
    t0 = time.perf_counter()
    out = c_port.remap(wl["out"], wl["rotations"], wl["src"], image, rows=rows, threads=0)
    dt = time.perf_counter() - t0
    return {"value": out.shape[0] * out.shape[1] / dt / 1e9, "unit": UNIT,
            "cores": len(os.sched_getaffinity(0)), "kind": "port",
            "sample": f"oracle/pb_oracle.c, one full {name} frame, {dt:.2f} s wall"}


# --------------------------------------------------------------------------------------------
# clocks


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs.
    NVML is initialised in the constructor (it takes longer than a short timed region), and
    ``start()`` returns only after the first sample is in."""

    def __init__(self, index: int, period: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self._first = threading.Event()
        self.error = None
        self._nv = self._handle = None
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nv = nv
            self._handle = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._handle, nv.NVML_CLOCK_SM)
            self._names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
        except Exception as exc:  # NVML missing: report it, never fake numbers
            self.error = repr(exc)

    def _sample(self):
        nv, h = self._nv, self._handle
        self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        for bit, nm in self._names.items():
            if mask & bit:
                self.reasons.add(nm)

    def run(self):
        if self._nv is None:
            self._first.set()
            return
        try:
            while not self._halt.is_set():
                self._sample()
                self._first.set()
                time.sleep(self.period)
        except Exception as exc:
            self.error = repr(exc)
            self._first.set()

    def start(self):
        super().start()
        self._first.wait(timeout=2)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        out = {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
               "samples": len(self.samples)}
        if self.error:
            out["error"] = self.error
        return out


# --------------------------------------------------------------------------------------------
# GPU arm


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except (ValueError, IndexError):
            pass
    return local_rank


def make_device_batch(torch, name, frames, rank):
    """``frames`` distinct synthetic frames of the workload, generated on the device from the
    workload's seed (+ global frame index); synthetic uniform noise like the parity inputs."""
    wl = workloads.WORKLOADS[name]
    src = wl["src"]
    gen = torch.Generator(device="cuda")
    gen.manual_seed((wl["seed"] or 1234) + 1000 * rank)
    return torch.randint(0, 256, (frames, src["height"], src["width"], CHANNELS), dtype=torch.uint8,
                         device="cuda", generator=gen)


def timed_kernel_steps(torch, source, cmap, batch, out, steps, warmup, dist, sampler=None, step_fn=None):
    from photonbend_b200.batch import remap_batch

    if step_fn is not None:
        def remap_batch(source, cmap, batch, out):  # noqa: F811  (one step = whatever step_fn does)
            step_fn()

    for _ in range(warmup):
        remap_batch(source, cmap, batch, out)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()  # clocks are sampled from here to the end of the timed region
    stream = torch.cuda.current_stream()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    t_begin = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    from photonbend_b200 import _native

    lib = _native.load()
    launches0 = lib.pb_kernel_launches()
    t_begin.record(stream)
    for k in range(steps):
        starts[k].record(stream)
        remap_batch(source, cmap, batch, out)
        ends[k].record(stream)
    t_end.record(stream)
    torch.cuda.synchronize()
    timed_kernel_steps.launches = lib.pb_kernel_launches() - launches0  # counted by the library itself
    if dist is not None:
        dist.barrier()
    total_ms = t_begin.elapsed_time(t_end)
    launch_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    return total_ms, launch_ms


def timed_e2e_steps(torch, source, cmap, name, frames, steps, warmup, dist, batch=4):
    """Public-API path with pinned host buffers; H2D + kernel + D2H of every frame timed.
    Every frame of a step has its own pinned output buffer (no two copies in flight share one);
    the inputs cycle over a small pool (they are only read)."""
    from photonbend_b200.batch import FramePipeline

    wl = workloads.WORKLOADS[name]
    src = wl["src"]
    oh, ow, _ = workloads.output_shape(wl["out"])
    pool = min(frames, 4)
    rng = np.random.default_rng(99)
    host_in = []
    for _ in range(pool):
        t = torch.empty((src["height"], src["width"], CHANNELS), dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = rng.integers(0, 256, t.shape, dtype=np.uint8)
        host_in.append(t)
    host_out = [torch.empty((oh, ow, CHANNELS), dtype=torch.uint8, pin_memory=True) for _ in range(frames)]
    pipe = FramePipeline(source, cmap, depth=3, batch=batch)

    def one_step():
        for k in range(frames):
            pipe.submit(host_in[k % pool], host_out[k])
        pipe.drain()

    for _ in range(max(1, min(warmup, 2))):
        one_step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    from photonbend_b200 import _native

    lib = _native.load()
    launches0 = lib.pb_kernel_launches()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if dist is not None:
        dist.barrier()
    h2d = frames * src["height"] * src["width"] * CHANNELS
    d2h = frames * oh * ow * CHANNELS
    return dt, h2d, d2h, lib.pb_kernel_launches() - launches0, host_in, host_out


def timed_compressed_stream(torch, source, cmap, name, frames, steps):
    """The same stream with JPEG bytes across PCIe instead of raw pixels (SURVEY section 8f.1 / f.3):
    nvJPEG decode on the device -> remap (8 frames per launch) -> nvJPEG encode on the device, through
    photonbend_b200.stream.remap_jpeg_stream on THIS rank's GPU.  The frames are smooth synthetic
    images (noise does not compress and is not what a camera delivers); bytes per step are counted
    from the bitstreams.  nvJPEG is a library codec -- plumbing either side of the hot path."""
    import io

    from PIL import Image

    from photonbend_b200 import stream

    wl = workloads.WORKLOADS[name]
    src = wl["src"]
    h, w = src["height"], src["width"]
    yy, xx = np.mgrid[0:h, 0:w]
    jpegs = []
    for k in range(min(frames, 4)):
        img = np.stack([(xx * (k + 1) // 8) % 256, (yy // 4 + 40 * k) % 256, ((xx + yy) // 16) % 256], axis=2).astype(np.uint8)
        buf = io.BytesIO()
        Image.fromarray(img).save(buf, format="JPEG", quality=90)
        jpegs.append(buf.getvalue())
    # one call carries 4 steps' worth of frames, so that the stream's pipeline (decode of batch n + 1
    # under remap + encode of batch n) is in steady state for most of the timed region
    reps = 4
    stream_in = [jpegs[k % len(jpegs)] for k in range(frames * reps)]
    dev = [torch.cuda.current_device()]
    out = stream.remap_jpeg_stream(source, cmap, stream_in[:frames], devices=dev, batch=8)  # warm-up (nvJPEG start-up, plan)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = stream.remap_jpeg_stream(source, cmap, stream_in, devices=dev, batch=8)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    from photonbend_b200.utils import image_io

    fallbacks = int(image_io.load_codec().pb_io_single_state_decodes())
    return dt, sum(len(j) for j in stream_in) // reps, sum(len(j) for j in out) // reps, fallbacks


DUMP_MAX_BYTES = 48 << 20  # --dump-outputs stays under 64 MB in all


def output_sample(torch, out):
    """What --dump-outputs writes for one uint8 output tensor (..., C): the whole tensor as float32
    when it fits DUMP_MAX_BYTES, else the channels of a fixed, seeded, sorted sample of its pixels
    as ``values`` (n, C) and their coordinates, one column per leading axis (frame, row, column),
    as ``pixels`` (float32 holds every index below 2^24 exactly)."""
    if out.numel() * 4 <= DUMP_MAX_BYTES:
        return {"": out.float().cpu().numpy()}
    shape = tuple(out.shape)
    flat = out.reshape(-1, shape[-1])
    n = DUMP_MAX_BYTES // (4 * (shape[-1] + len(shape) - 1))
    idx = np.sort(np.random.default_rng(0).choice(flat.shape[0], n, replace=False))
    values = flat[torch.from_numpy(idx).to(out.device)].float().cpu().numpy()
    pixels = np.stack(np.unravel_index(idx, shape[:-1]), axis=1).astype(np.float32)
    return {"_values": values, "_pixels": pixels}


def dump_outputs(directory, name, sample):
    os.makedirs(directory, exist_ok=True)
    for suffix, array in sample.items():
        np.save(os.path.join(directory, f"{name}{suffix}.npy"), array)
    log(f"[bench] wrote {', '.join(name + s + '.npy' for s in sample)} to {directory}")


def parity_check(name, pairs):
    """Bit-compare remapped frames with the CPU oracle (oracle/pb_oracle.c on all cores; it is
    sha256-identical to the reference at full size, tests/golden).  pairs: (source HWC uint8
    ndarray, output ndarray).  The checker runs after the timed regions, never inside them."""
    from oracle import c_port

    wl = workloads.WORKLOADS[name]
    bad = 0
    for image, got in pairs:
        want = c_port.remap(wl["out"], wl["rotations"], wl["src"], image)
        bad += int((want != got).any(axis=2).sum())
    return {"checked_frames": len(pairs), "mismatch_px": bad,
            "checker": "oracle/pb_oracle.c (sha256-identical to the reference on this geometry)"}


def graph_launch_ms(torch, source, cmap, pool, outs, launches=20, replays=7):
    """Average duration of ONE launch when ``launches`` of them run back to back as a CUDA graph
    (events around the replay): for kernels of a few tens of microseconds, events around a single
    launch also time the host's way from the first event to the launch (Python, ctypes, the plan's
    mutex: ~10 us on a cold host core), a graph does not.  Launch k works on frame k mod len(pool):
    the pool is larger than L2, so no launch finds its source or its output in the cache.
    None if the capture is refused."""
    from photonbend_b200.batch import remap_batch

    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for k in range(len(pool)):
                remap_batch(source, cmap, pool[k], outs[k])
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for k in range(launches):
                remap_batch(source, cmap, pool[k % len(pool)], outs[k % len(pool)])
        graph.replay()
        torch.cuda.synchronize()
        times = []
        for _ in range(replays):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / launches)
        return float(np.median(times))
    except Exception as exc:  # noqa: BLE001
        log(f"[bench] CUDA graph timing unavailable: {exc!r}")
        return None


def quick_kernel_rate(torch, name, frames, steps=20, warmup=3):
    """Kernel-only Gpix/s + roofline of another workload (reported under "also")."""
    import helpers
    from photonbend_b200.batch import remap_batch

    wl = workloads.WORKLOADS[name]
    info = golden_info(name)
    # one frame per launch: a pool of distinct frames and outputs larger than 2 x L2, cycled, so that
    # no launch finds its data in the 126 MB L2 (a batch of 16 frames is larger than L2 by itself)
    n_pool = 1
    if frames == 1:
        per_launch = (info["src_pixels"] + info["out_pixels"]) * CHANNELS
        n_pool = max(2, -(-(2 * 126 * 1024 * 1024) // per_launch) + 1)
    batch = make_device_batch(torch, name, frames * n_pool, 0)
    source = helpers.product_image(wl["src"], batch[:frames])
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    pool = [batch[k * frames:(k + 1) * frames] for k in range(n_pool)]
    outs = [remap_batch(source, cmap, p) for p in pool]
    state = {"k": 0}

    def step():
        k = state["k"] = (state["k"] + 1) % n_pool
        remap_batch(source, cmap, pool[k], outs[k])

    total_ms, launch_ms = timed_kernel_steps(torch, source, cmap, None, None, steps, warmup, None, step_fn=step)
    px = info["out_pixels"] * frames
    events_ms = float(np.median(launch_ms))
    avg_ms, statistic = events_ms, "median of 20 launches, events around each launch"
    if frames == 1:
        graph_ms = graph_launch_ms(torch, source, cmap, pool, outs)
        if graph_ms is not None:
            avg_ms = graph_ms
            statistic = (f"20 launches replayed back to back as one CUDA graph over a pool of {n_pool} frames "
                         "(larger than 2 x L2), events around the replay, median of 7")
    peak, _ = measured_peak_gbs()
    achieved = algorithmic_bytes_per_frame(name) * frames / (avg_ms * 1e-3) / 1e9
    del batch, outs, pool
    torch.cuda.empty_cache()
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": committed_traffic(name, frames)}
    extra = committed_counters(name, frames)
    if wl["rotations"]:
        # one frame through a rotated geometry is bound by instruction issue / the FP64 pipe (the
        # per-pixel float64 resolve), not by HBM: the HBM fraction is reported for completeness
        roof["bound"] = "issue/fp64"
    if extra:
        roof.update(extra)
    return {"title": wl["title"], "frames_per_launch": frames, "value": px / (avg_ms * 1e-3) / 1e9,
            "unit": UNIT, "ms_per_launch": avg_ms, "statistic": statistic,
            "ms_per_launch_events_around_each": events_ms, "roofline": roof}


def run_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    name = args.workload

    cpu = None
    cport = None
    if world == 1 and not args.no_cpu_baseline:
        # before CUDA is initialised in this process: the CPU arm forks worker processes
        log(f"[bench] timing the CPU reference arm on {len(os.sched_getaffinity(0))} cores ...")
        cpu = cpu_baseline(name, budget_s=args.cpu_budget)
        cport = c_port_rate(name)

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        # stdout carries ONE JSON line: keep NCCL's version banner (NCCL_DEBUG=VERSION) off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod

    import helpers
    from photonbend_b200.batch import remap_batch

    wl = workloads.WORKLOADS[name]
    frames = args.frames
    batch = make_device_batch(torch, name, frames, rank)
    source = helpers.product_image(wl["src"], batch)
    cmap = helpers.product_map(wl["out"], wl["rotations"])
    out = remap_batch(source, cmap, batch)
    torch.cuda.synchronize()

    if args.shard == "rows":
        return run_gpu_rows(args, torch, dist, rank, local_rank, world, batch, source, cmap, cpu)

    sampler = ClockSampler(physical_gpu_index(local_rank))
    total_ms, launch_ms = timed_kernel_steps(torch, source, cmap, batch, out, args.steps, args.warmup, dist, sampler)
    clocks = sampler.stop()
    gpu_launches = timed_kernel_steps.launches
    dumped = output_sample(torch, out) if args.dump_outputs else None

    # the same steps back to back for >= --sustain-seconds: the K steps above are a burst of a few
    # milliseconds; this is what the kernel holds once the power limit has had time to act
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / max(total_ms / args.steps, 1e-3)) + 1)
        sampler2 = ClockSampler(physical_gpu_index(local_rank))
        sus_ms, sus_launch_ms = timed_kernel_steps(torch, source, cmap, batch, out, n_sus, 0, dist, sampler2)
        sustained = {"steps": n_sus, "total_ms": sus_ms, "launch_ms": float(np.mean(sus_launch_ms)),
                     "clocks": sampler2.stop()}

    e2e_dt, h2d, d2h, e2e_launches, host_in, host_out = timed_e2e_steps(
        torch, source, cmap, name, frames, max(1, args.e2e_steps), args.warmup, dist, batch=args.e2e_batch)
    # the same stream with four frames per launch (the batched kernel): fewer, larger launches --
    # the copies, not the kernel, bound a host-resident stream, so this is reported, not the headline
    e2e_other = None
    if world == 1 and args.e2e_batch == 1 and frames >= 4:
        dt4, _, _, l4, _, _ = timed_e2e_steps(torch, source, cmap, name, frames, 1, 1, dist, batch=4)
        e2e_other = (dt4, l4)

    compressed = None
    if not args.no_compressed:
        try:
            c_dt, c_up, c_down, c_single = timed_compressed_stream(torch, source, cmap, name, frames, 1)
            compressed = [c_dt, c_up, c_down, c_single]
        except Exception as exc:  # the codec library is optional plumbing: say why, keep the line
            compressed = repr(exc)

    # parity of what was just timed (after the timed regions; rank 0's frames): frames of the
    # device batch as the last timed step left them, and host frames that went through the pipeline
    parity = None
    if rank == 0 and not args.no_parity:
        pairs = [(batch[k].cpu().numpy(), out[k].cpu().numpy()) for k in sorted({0, frames - 1})]
        pool = len(host_in)
        pairs += [(host_in[k % pool].numpy(), host_out[k].numpy()) for k in sorted({1 % frames, frames - 1})]
        parity = parity_check(name, pairs)
        parity["what"] = (f"{len(pairs) - 2 if frames > 1 else 1} frame(s) of the timed device batch (`value`) and 2 host frames of the "
                          "last end-to-end step (`e2e`), whole frames, bit for bit")

    from photonbend_b200.batch import max_over_ranks

    timings = [total_ms, e2e_dt * 1e3, compressed[0] * 1e3 if isinstance(compressed, list) else 0.0] + (
        [sustained["total_ms"]] if sustained else [])
    timings = max_over_ranks(timings, device="cuda")  # timing only
    total_ms, e2e_ms, comp_ms = timings[0], timings[1], timings[2]
    timings = timings[:2] + timings[3:]

    info = golden_info(name)
    px_per_step = info["out_pixels"] * frames * world
    ms_per_step = total_ms / args.steps
    value = px_per_step / (ms_per_step * 1e-3) / 1e9
    e2e_value = px_per_step * max(1, args.e2e_steps) / (e2e_ms * 1e-3) / 1e9

    peak, peak_src = measured_peak_gbs()
    avg_launch_ms = float(np.mean(launch_ms))
    achieved = algorithmic_bytes_per_frame(name) * frames / (avg_launch_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": args.traffic_bytes if args.traffic_bytes is not None else committed_traffic(name, frames),
        "traffic_source": "ncu --set full capture of one launch, profiles/traffic.json", "peak_source": peak_src,
        "kernel": ("pb::remap_tiled_kernel, %d grid(s) per step (a double-fisheye source is remapped as two grids of "
                   "the same kernel, one per tile class; launch_ms, achieved and traffic cover both)"
                   % max(1, gpu_launches // max(1, args.steps))),
        "launch_ms": avg_launch_ms,
        "algorithmic_bytes_per_launch": algorithmic_bytes_per_frame(name) * frames,
    }

    if sustained:
        sus_ms_per_step = timings[2] / sustained["steps"]
        sustained.update({
            "value": px_per_step / (sus_ms_per_step * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": sus_ms_per_step,
            "seconds": timings[2] * 1e-3,
            "roofline_frac": algorithmic_bytes_per_frame(name) * frames / (sustained["launch_ms"] * 1e-3) / 1e9 / peak})
        del sustained["total_ms"]

    also = {}
    if world == 1 and not args.no_also:
        for other, fr in (("T", frames), ("T", 1), ("cfg1", 1), ("cfg2", 1), ("cfg3", 1), ("cfg4", 1)):
            if other != name:
                also[other if (fr == 1) == (other != "T") else f"{other}_{fr}frame"] = quick_kernel_rate(torch, other, fr)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "dtype_note": "float64 index arithmetic on uint8 pixels",
            "data": "synthetic uniform-noise uint8 frames (seeded), generated on device",
            "config": bench_config(name, frames),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": f"photonbend_b200.batch.FramePipeline (pinned host frames in and out, depth 3, "
                           f"{args.e2e_batch} frames per launch)",
                    "steps": max(1, args.e2e_steps)},
            "gpu_launches": gpu_launches,
            "e2e_gpu_launches": e2e_launches,
            "clocks": clocks,
            "roofline": roofline,
        }
        if e2e_other is not None:
            line["e2e"]["four_frames_per_launch"] = {"value": px_per_step / e2e_other[0] / 1e9, "unit": UNIT,
                                                     "gpu_launches": e2e_other[1]}
        if isinstance(compressed, list):
            line["e2e_compressed"] = {
                "value": px_per_step / (comp_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": compressed[1],
                "d2h_bytes_per_step": compressed[2], "single_state_decodes": compressed[3],
                "api": "photonbend_b200.stream.remap_jpeg_stream: JPEG bytes in, nvJPEG decode + remap (8 frames per "
                       "launch) + nvJPEG encode on the device, JPEG bytes out; smooth synthetic frames, quality 90 in / 75 out; "
                       "one call over 4 steps' worth of frames",
                "note": "bounded by the nvJPEG library codec (decoupled decoder, Huffman stage on the device, up to 8 decode threads per GPU), not by the remap kernel or PCIe"}
        elif compressed is not None:
            line["e2e_compressed"] = {"unavailable": compressed}
        if sustained:
            line["sustained"] = sustained
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            cpu["c_port_all_cores"] = cport
            line["cpu_baseline"] = cpu
        if also:
            line["also"] = also
        emit_line(line)
    if dumped is not None:
        dump_outputs(args.dump_outputs, "out" if world == 1 else f"out_rank{rank}", dumped)
    if dist is not None:
        dist.destroy_process_group()


def run_gpu_rows(args, torch, dist, rank, local_rank, world, batch, source, cmap, cpu):
    """--shard rows: every frame of the step is cut into ``world`` output-row bands, one per GPU
    (batch.shard_rows / remap_row_band -> pb_plan_remap_rows_u8); every GPU holds the whole source
    frames, nothing is exchanged.  Total work is fixed as N grows: strong scaling.  Device-resident
    only (the bands stay on the GPUs that made them)."""
    from photonbend_b200 import _native
    from photonbend_b200.batch import max_over_ranks, remap_row_band, shard_rows

    name, frames = args.workload, args.frames
    info = golden_info(name)
    oh, ow = info["shape"][0], info["shape"][1]
    rows = shard_rows(oh, rank, world)
    bands = torch.empty((frames, max(1, len(rows)), ow, CHANNELS), dtype=torch.uint8, device="cuda")

    def step():
        if len(rows) > 0:
            for f in range(frames):
                remap_row_band(source, cmap, batch[f], rows, bands[f])

    sampler = ClockSampler(physical_gpu_index(local_rank))
    total_ms, launch_ms = timed_kernel_steps(torch, source, cmap, batch, None, args.steps, args.warmup, dist, sampler, step_fn=step)
    clocks = sampler.stop()
    gpu_launches = timed_kernel_steps.launches
    if args.dump_outputs and len(rows) > 0:
        dump_outputs(args.dump_outputs, "bands" if world == 1 else f"bands_rank{rank}", output_sample(torch, bands))
    (total_ms,) = max_over_ranks([total_ms], device="cuda")
    ms_per_step = total_ms / args.steps
    px_per_step = info["out_pixels"] * frames
    value = px_per_step / (ms_per_step * 1e-3) / 1e9
    peak, peak_src = measured_peak_gbs()
    achieved = algorithmic_bytes_per_frame(name) * frames / (ms_per_step * 1e-3) / 1e9
    parity = None
    if rank == 0 and not args.no_parity and len(rows) > 0:
        from oracle import c_port

        wl = workloads.WORKLOADS[name]
        want = c_port.remap(wl["out"], wl["rotations"], wl["src"], batch[0].cpu().numpy(), rows=(rows.start, rows.stop))
        parity = {"checked_frames": 1, "mismatch_px": int((want != bands[0].cpu().numpy()).any(axis=2).sum()),
                  "what": f"rank 0's band (rows {rows.start}..{rows.stop}) of frame 0 against oracle/pb_oracle.c"}
    if rank == 0:
        cfg = bench_config(name, frames)
        cfg["sharding"] = f"output-row bands of every frame over {world} GPU(s) (tile-aligned), whole source on every GPU, no collective"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic uniform-noise uint8 frames (seeded), generated on device",
            "config": cfg, "gpu_launches": gpu_launches, "clocks": clocks,
            "e2e": None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                         "frac": achieved / (peak * world), "traffic": None, "peak_source": peak_src + f" x {world} GPUs",
                         "kernel": "single-frame kernels over a row band (pb_plan_remap_rows_u8), one launch per frame and GPU"},
        }
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            line["cpu_baseline"] = cpu
        emit_line(line)
    if dist is not None:
        dist.destroy_process_group()


def run_reference(args):
    """--impl reference: the reference's own CPU implementation on all host cores (see CpuArm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    arm = CpuArm(name)
    # size one step so that steps + warmup end within a few minutes
    per_step_s = max(0.5, args.cpu_budget * 8 / (args.steps + args.warmup))
    rows = arm.pick_band_rows(per_step_s)
    for _ in range(args.warmup):
        arm.step(rows)
    tot_px, tot_dt, match = 0, 0.0, None
    for _ in range(args.steps):
        px, dt, out = arm.step(rows)
        tot_px += px
        tot_dt += dt
        if match is None:
            match = arm.whole_frame_matches_golden(out)
    value = tot_px / tot_dt / 1e9
    cpu = {"value": value, "unit": UNIT, "cores": arm.procs, "kind": arm.kind,
           "sample": arm.describe(rows, tot_px, tot_dt, args.steps)}
    if match is not None:
        cpu["output_sha256_matches_reference_golden"] = bool(match)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "dtype_note": "float64 index arithmetic on uint8 pixels",
        "data": "synthetic uniform-noise uint8 frame (seeded)",
        "config": bench_config(name, args.frames),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)


_RESULT_FD = None


def claim_stdout():
    """stdout carries ONE JSON line: everything else that writes to fd 1 (NCCL's version banner,
    library chatter of child processes) goes to stderr from here on."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(workloads.WORKLOADS))
    ap.add_argument("--frames", type=int, default=16, help="frames per step per GPU (one launch)")
    ap.add_argument("--shard", default="frames", choices=["frames", "rows"],
                    help="frames: every GPU remaps its own frames (weak scaling, the default); rows: every frame is "
                         "cut into output-row bands, one per GPU (strong scaling, device-resident)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-batch", type=int, default=1, help="frames per launch of the end-to-end pipeline")
    ap.add_argument("--sustain-seconds", type=float, default=1.5,
                    help="also time the same steps back to back for at least this long (0 = off)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed outputs")
    ap.add_argument("--no-compressed", action="store_true", help="skip the compressed-stream (nvJPEG) end-to-end leg")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU-arm wall time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed to DIR/<name>.npy as float32 "
                         "(a fixed, seeded sample of its pixels when the output is larger than 48 MB as float32); "
                         "the synthetic inputs depend on the arguments only, so two builds can be compared. "
                         "GPU path only: a step of --impl reference covers row bands whose height is chosen "
                         "from a timing, so its output differs from run to run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: a step of --impl reference covers row bands sized from a "
                 "timing, so what it computes is not the same from run to run")
    claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
