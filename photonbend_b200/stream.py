"""Image FILES that share one geometry (the frames of a video dumped to a directory, a batch of
photos from one camera): decode -> remap -> encode, sharded over the GPUs of the box.

The reference has no such entry point: its commands convert one file per process
(photonbend/scripts/commands/make_pano.py:94-139 and twins).  Here the three commands accept a
DIRECTORY as input (and output): frame k goes to GPU k mod G (``batch.shard_frames``; no exchange
between GPUs), every GPU runs a ``batch.FramePipeline`` (pinned host buffers, copies and kernels of
neighbouring frames overlapped) fed by a small pool of codec threads.

Two codecs, as for single files (``utils/image_io.py``):

* ``pil``     Pillow on the host, like the reference: raw frames cross PCIe (88 MB each way for 8K);
* ``nvjpeg``  compressed stream: JPEG bytes go up, are decoded on the device (nvJPEG) into the batch
              buffer the remap kernel reads, the remapped frames are encoded on the device and JPEG
              bytes come back -- PCIe carries ~10x fewer bytes.  Not bit-identical to Pillow's codec.
"""

from __future__ import annotations

import os
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import List, Optional, Sequence

import numpy as np

from photonbend_b200 import engine
from photonbend_b200.batch import FramePipeline, shard_frames
from photonbend_b200.core.coordinate_map import CoordinateMap
from photonbend_b200.utils import image_io

IMAGE_SUFFIXES = (".jpg", ".jpeg", ".png")


def list_frames(directory) -> List[Path]:
    """Image files of a directory, sorted by name (the frame order)."""
    return sorted(p for p in Path(directory).iterdir() if p.is_file() and p.suffix.lower() in IMAGE_SUFFIXES)


def _decode_host(path) -> np.ndarray:
    from PIL import Image

    with Image.open(path) as img:
        return np.asarray(img)


def _encode_host(pixels: np.ndarray, path) -> None:
    from PIL import Image

    Image.fromarray(pixels).save(path)


def _host_worker(device: int, frames: Sequence[int], source, cmap, in_files, out_files, depth, batch, codec_threads, shape,
                 rotations=None):
    """Pillow codec: pinned host frames through a FramePipeline on GPU ``device`` (frame k through
    ``rotations[k]`` when given)."""
    torch = engine._torch()
    with torch.cuda.device(device):
        pipe = FramePipeline(source, cmap, depth=depth, device=device, batch=batch)
        oh, ow = pipe.output_shape
        window = (depth + 1) * batch
        ins = [torch.empty(shape, dtype=torch.uint8, pin_memory=True) for _ in range(window)]
        outs = [torch.empty((oh, ow) + tuple(shape[2:]), dtype=torch.uint8, pin_memory=True) for _ in range(window)]
        encoding = [None] * window      # encode future still reading outs[slot]
        launch_of = [None] * window     # index of the launch that carries the slot's frame
        launches = []                   # [event, [(slot, frame), ...]] in submission order
        retired = 0
        with ThreadPoolExecutor(max_workers=codec_threads) as pool:
            ahead = min(window, len(frames))
            decoded = {frames[n]: pool.submit(_decode_host, in_files[frames[n]]) for n in range(ahead)}

            def retire(upto):
                nonlocal retired
                while retired < upto:
                    event, group = launches[retired]
                    event.synchronize()
                    for s, k in group:
                        encoding[s] = pool.submit(_encode_host, outs[s].numpy(), out_files[k])
                    retired += 1

            group = []
            for n, k in enumerate(frames):
                slot = n % window
                if launch_of[slot] is not None:
                    retire(launch_of[slot] + 1)
                if encoding[slot] is not None:
                    encoding[slot].result()
                    encoding[slot] = None
                pixels = decoded.pop(k).result()
                if n + ahead < len(frames):
                    nxt = frames[n + ahead]
                    decoded[nxt] = pool.submit(_decode_host, in_files[nxt])
                if tuple(pixels.shape) != tuple(shape):
                    raise ValueError(f"{in_files[k]}: shape {pixels.shape} differs from the first frame's {tuple(shape)}")
                ins[slot].numpy()[...] = pixels
                group.append((slot, k))
                launch_of[slot] = len(launches)
                event = pipe.submit(ins[slot], outs[slot], None if rotations is None else rotations[k])
                if event is not None:
                    launches.append([event, group])
                    group = []
            event = pipe.flush()
            if event is not None:
                launches.append([event, group])
            retire(len(launches))
            for fut in encoding:
                if fut is not None:
                    fut.result()
        return pipe.kernel_launches


def _default_decode_threads(batch: int, n_devices: int) -> int:
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # (per GPU: the producer, the consumer and the decode threads; half of what is left of this GPU's share of the cores)
    return max(1, min(8, batch, (cores // max(1, n_devices) - 2) // 2 + 1))


def _compressed_pipeline(device: int, frames: Sequence[int], source, cmap, load, store, batch: int, decode_threads: int,
                         shape, rotations=None) -> int:
    """Frames ``frames`` on GPU ``device``, compressed on both sides of PCIe: ``load(k)`` gives the JPEG
    bytes of frame k, ``store(k, data)`` takes the JPEG bytes of its remap.  A producer (the calling
    thread) has batch n + 1 decoded into the other of two device buffers by ``decode_threads``
    workers -- one frame each, every worker its own decoder state and stream -- while a consumer
    thread remaps batch n (ONE launch; frame k through ``rotations[k]`` when given) and encodes it.
    Returns the number of kernel launches."""
    torch = engine._torch()
    chunks = [frames[c0:c0 + batch] for c0 in range(0, len(frames), batch)]
    if not chunks:
        return 0
    with torch.cuda.device(device):
        rays, geom = cmap.rays, source._source_geometry()
        srcs = [torch.empty((batch,) + tuple(shape), dtype=torch.uint8, device=f"cuda:{device}") for _ in range(2)]
        dst = torch.empty((batch, rays.out.height, rays.out.output_width, shape[2]), dtype=torch.uint8,
                          device=f"cuda:{device}")
        decoded = [threading.Semaphore(0), threading.Semaphore(0)]  # buffer b holds a decoded batch
        free = [threading.Semaphore(1), threading.Semaphore(1)]     # buffer b may be overwritten
        failed: list = []
        consumer_stream = torch.cuda.Stream(device=device)

        def consume():
            try:
                with torch.cuda.device(device), torch.cuda.stream(consumer_stream):
                    for n, chunk in enumerate(chunks):
                        b = n & 1
                        decoded[b].acquire()
                        if failed:
                            return
                        k = len(chunk)
                        if rotations is not None:
                            engine.remap_frames_device(rays, geom, srcs[b][:k], [rotations[f] for f in chunk], dst[:k])
                        elif k == 1:
                            engine.remap_device(rays, geom, srcs[b][0], dst[0])
                        else:
                            engine.remap_device(rays, geom, srcs[b][:k], dst[:k])
                        torch.cuda.current_stream().synchronize()
                        free[b].release()  # the remap has read the batch: it may be decoded over
                        for i, f in enumerate(chunk):
                            store(f, image_io.encode_jpeg_from_device(dst[i]))
            except BaseException as exc:  # noqa: BLE001
                failed.append(exc)
                for sem in free:
                    sem.release()

        tls = threading.local()

        def decode_one(f, b, i):
            if not hasattr(tls, "stream"):
                tls.stream = torch.cuda.Stream(device=device)
            with torch.cuda.device(device), torch.cuda.stream(tls.stream):
                image_io.decode_jpeg_into(load(f), srcs[b][i])  # (synchronises its stream)

        consumer = threading.Thread(target=consume)
        consumer.start()
        try:
            with ThreadPoolExecutor(max_workers=decode_threads) as pool:
                for n, chunk in enumerate(chunks):
                    b = n & 1
                    free[b].acquire()
                    if failed:
                        break
                    for fut in [pool.submit(decode_one, f, b, i) for i, f in enumerate(chunk)]:
                        fut.result()
                    decoded[b].release()
        except BaseException as exc:  # noqa: BLE001
            failed.append(exc)
            for sem in decoded:
                sem.release()
        consumer.join()
        if failed:
            raise failed[0]
    return len(chunks)


def _device_worker(device: int, frames: Sequence[int], source, cmap, in_files, out_files, batch, shape, n_devices=1,
                   rotations=None):
    """nvJPEG codec on files: compressed bytes up, decode -> remap -> encode on GPU ``device``, compressed bytes down."""

    def load(k):
        with open(in_files[k], "rb") as fh:
            return fh.read()

    def store(k, data):
        with open(out_files[k], "wb") as fh:
            fh.write(data)

    if batch <= 1:
        batch = 8  # (frames of a batch are decoded at once; one frame per launch would decode one at a time)
    return _compressed_pipeline(device, frames, source, cmap, load, store, batch, _default_decode_threads(batch, n_devices), shape,
                                rotations)


def _frame_rotations(frame_rotations, n_frames: int):
    """(N, 3, 3) float64 matrices of per-frame rotations, checked against the number of frames; None stays None."""
    if frame_rotations is None:
        return None
    mats = engine.frame_matrices(frame_rotations).reshape(-1, 3, 3)
    if mats.shape[0] != n_frames:
        raise ValueError(f"{mats.shape[0]} frame rotations for {n_frames} frames")
    return mats


def remap_jpeg_stream(source, coordinate_map: CoordinateMap, jpegs: Sequence[bytes], devices: Optional[Sequence[int]] = None,
                      batch: int = 8, decode_threads: Optional[int] = None, frame_rotations=None) -> List[bytes]:
    """Compressed stream in memory: JPEG bytes in -> nvJPEG decode on the device -> ONE remap launch
    per ``batch`` frames -> nvJPEG encode on the device -> JPEG bytes out.  Frame k on GPU
    ``devices[k mod G]``; per GPU a producer that decodes batch k + 1 with ``decode_threads`` host
    threads (each its own decoder state and stream; default: up to 8, at most one per frame of a
    batch and what the host's cores allow per GPU) while a consumer remaps and encodes batch k; raw
    pixels never cross PCIe.  ``frame_rotations``: one rotation per frame, as in ``remap_files``."""
    if not (isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy):
        raise ValueError("remap_jpeg_stream needs the lazy CoordinateMap of get_coordinate_map()")
    rotations = _frame_rotations(frame_rotations, len(jpegs))
    torch = engine._torch()
    if devices is None:
        devices = list(range(torch.cuda.device_count()))
    devices = list(devices)[: max(1, len(jpegs))]
    if decode_threads is None:
        decode_threads = _default_decode_threads(batch, len(devices))
    shape = tuple(source.image.shape)[-3:]  # (H, W, C) of one frame (the image may be a batch)
    out: List[Optional[bytes]] = [None] * len(jpegs)
    errors = []

    def store(k, data):
        out[k] = data

    def run(g):
        try:
            frames = list(shard_frames(len(jpegs), g, len(devices)))
            _compressed_pipeline(devices[g], frames, source, coordinate_map, jpegs.__getitem__, store, batch,
                                 decode_threads, shape, rotations)
        except BaseException as exc:  # noqa: BLE001
            errors.append(exc)

    threads = [threading.Thread(target=run, args=(g,)) for g in range(len(devices))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return out  # type: ignore[return-value]


def remap_files(source, coordinate_map: CoordinateMap, in_files: Sequence, out_files: Sequence,
                devices: Optional[Sequence[int]] = None, depth: int = 3, batch: int = 1,
                codec: Optional[str] = None, codec_threads: int = 4, frame_rotations=None) -> dict:
    """Remap ``in_files[k]`` -> ``out_files[k]`` for files that all have the geometry of ``source``
    (a CameraImage / DoubleCameraImage / PanoramaImage; its own ``image`` only gives the frame
    shape) along the lazy ``coordinate_map``.  Frame k runs on ``devices[k mod G]`` (default: every
    visible GPU), one host thread per GPU.  ``frame_rotations`` (one ``Rotation`` or 3x3 matrix per
    file): frame k is remapped as if ``frame_rotations[k]`` had been applied after the map's own
    rotations, and the rotation travels with the frame to its GPU.  Returns {"frames", "gpus",
    "seconds", "kernel_launches"}."""
    if not (isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy):
        raise ValueError("remap_files needs the lazy CoordinateMap of get_coordinate_map()")
    if len(in_files) != len(out_files):
        raise ValueError("in_files and out_files differ in length")
    rotations = _frame_rotations(frame_rotations, len(in_files))
    torch = engine._torch()
    codec = codec or image_io.selected_codec()
    if devices is None:
        devices = list(range(torch.cuda.device_count()))
    devices = list(devices)[: max(1, len(in_files))]
    shape = tuple(source.image.shape)[-3:]  # (H, W, C) of one frame
    on_device = codec == "nvjpeg" and len(shape) == 3 and shape[2] == 3 and all(
        Path(p).suffix.lower() in (".jpg", ".jpeg") for p in list(in_files) + list(out_files))
    results, errors = [0] * len(devices), []

    def run(g):
        frames = list(shard_frames(len(in_files), g, len(devices)))
        try:
            if on_device:
                results[g] = _device_worker(devices[g], frames, source, coordinate_map, in_files, out_files, max(1, batch), shape,
                                            len(devices), rotations)
            else:
                results[g] = _host_worker(devices[g], frames, source, coordinate_map, in_files, out_files, depth,
                                          max(1, batch), codec_threads, shape, rotations)
        except BaseException as exc:  # noqa: BLE001  (re-raised on the calling thread)
            errors.append(exc)

    t0 = time.perf_counter()
    threads = [threading.Thread(target=run, args=(g,)) for g in range(len(devices))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return {"frames": len(in_files), "gpus": len(devices), "seconds": time.perf_counter() - t0,
            "kernel_launches": sum(results), "codec": "nvjpeg" if on_device else "pil"}
