"""Frame streams: many frames that share one geometry (a video, BASELINE config 5).

The reference has no such entry point -- its commands remap one image per process.  Two things
make a stream cheap on a B200:

* the source index of an output pixel depends on the geometry only, so one launch resolves it
  once and applies it to every frame of a device batch (``pb_remap_u8`` with n_frames > 1);
* host <-> device copies of neighbouring frames overlap with each other and with the kernel
  when they are issued on separate CUDA streams from pinned memory (``FramePipeline``).

Sharding over the GPUs of a box needs no collective: frame k goes to GPU k mod G
(``shard_frames``), every GPU owns its inputs and outputs.  A single large frame can instead be
cut into output-row bands (``shard_rows`` + ``remap_row_band``): every GPU holds the whole source
and produces its band.
"""

from __future__ import annotations

from typing import List, Optional, Sequence

from photonbend_b200 import engine
from photonbend_b200.core.coordinate_map import CoordinateMap


def shard_frames(n_frames: int, rank: int, world_size: int) -> range:
    """Indices of the frames rank ``rank`` of ``world_size`` processes: k = rank (mod world_size).
    Round-robin keeps every GPU's share within one frame of the others for any stream length."""
    if not 0 <= rank < world_size:
        raise ValueError(f"rank {rank} outside world of size {world_size}")
    return range(rank, n_frames, world_size)


ROW_BAND_ALIGN = 64  # rows of one output tile: bands that start on a tile row take the TMA-staged kernels


def shard_rows(height: int, rank: int, world_size: int, align: int = ROW_BAND_ALIGN) -> range:
    """Output rows of rank ``rank`` when ONE frame of ``height`` rows is cut into ``world_size``
    contiguous bands whose first rows are multiples of ``align`` (the last band takes what is
    left; ranks beyond the number of aligned bands get an empty range).  Every GPU needs the whole
    source; nothing is exchanged."""
    if not 0 <= rank < world_size:
        raise ValueError(f"rank {rank} outside world of size {world_size}")
    units = -(-height // align)                       # tile rows in the image
    lo = (units * rank) // world_size * align
    hi = (units * (rank + 1)) // world_size * align
    return range(min(lo, height), min(hi, height))


def remap_row_band(source, coordinate_map: CoordinateMap, frame, rows: range, out=None):
    """Rows ``rows`` (a contiguous range) of the remap of ONE device frame: the band alone, as a
    (len(rows), Wo, C) CUDA tensor of the frame's dtype.  ``frame`` is the whole source image on
    this device."""
    if not (isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy):
        raise ValueError("remap_row_band needs the lazy CoordinateMap of get_coordinate_map()")
    if rows.step != 1:
        raise ValueError("a band is a contiguous range of rows")
    return engine.remap_rows_device(coordinate_map.rays, source._source_geometry(), frame.contiguous(),
                                    rows.start, max(rows.start, rows.stop), out)


def max_over_ranks(values, device="cpu"):
    """Element-wise max of a list of floats over all ranks of the default process group (a
    timing reduction only -- the remap itself exchanges nothing between GPUs)."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.cpu()]


def remap_batch(source, coordinate_map: CoordinateMap, frames, out=None, frame_rotations=None):
    """Remap a device batch ``frames`` (CUDA tensor (N, H, W, C) of any dtype the remap takes, see
    ``engine.ELEM_BYTES``) that shares the geometry
    of ``source`` (a CameraImage / DoubleCameraImage / PanoramaImage whose own ``image`` is only
    used for its shape) along ``coordinate_map``.  One kernel launch; returns the (N, Ho, Wo, C)
    CUDA tensor of the same dtype.

    ``frame_rotations`` (N ``Rotation`` objects or an (N, 3, 3) array): frame k is remapped as if
    ``frame_rotations[k]`` had been applied to ``coordinate_map`` after its own rotations
    (stabilised or levelled video, a moving virtual camera)."""
    if not (isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy):
        raise ValueError("remap_batch needs the lazy CoordinateMap of get_coordinate_map()")
    if frames.dim() != 4 or not frames.is_cuda:
        raise ValueError("frames must be a CUDA tensor of shape (N, H, W, C)")
    if frame_rotations is not None:
        return engine.remap_frames_device(coordinate_map.rays, source._source_geometry(), frames.contiguous(),
                                          frame_rotations, out)
    return engine.remap_device(coordinate_map.rays, source._source_geometry(), frames.contiguous(), out)


class FramePipeline:
    """Host frames in, host frames out, with ``depth`` launches in flight.

    Slot s owns a device input buffer and a device output buffer for ``batch`` frames and a CUDA
    stream; frames fill the slots in turn.  The H2D copy of a frame is enqueued on its slot's
    stream as soon as it is submitted; when the slot holds ``batch`` frames (or on ``flush()`` /
    ``drain()``) ONE remap launch covers them -- the source index of an output pixel is resolved
    once per launch, not once per frame -- followed by their D2H copies.  Copies of one slot
    overlap the kernel and the copies of the others.  Host buffers should be pinned
    (``torch.empty(..., pin_memory=True)``) or the copies serialise.  ``batch=1`` launches per
    frame (lowest latency); a stream of frames wants ``batch`` >= 4.

    A host output buffer is complete after ``drain()`` or after the event its ``submit`` /
    ``flush`` returned; it must not be handed to another ``submit`` before that.

    ``submit(..., rotation=R)`` remaps that frame as if ``R`` had been applied after the map's own
    rotations (see ``remap_batch``'s ``frame_rotations``).  A pipeline takes a rotation with every
    frame or with none: an identity rotation is not bit-identical to no rotation (it sends each
    ray through acos / atan2 once more), so mixing the two would silently change some frames.
    """

    def __init__(self, source, coordinate_map: CoordinateMap, depth: int = 3, device: Optional[int] = None,
                 batch: int = 1):
        if not (isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy):
            raise ValueError("FramePipeline needs the lazy CoordinateMap of get_coordinate_map()")
        torch = engine._torch()
        self._torch = torch
        self._rays = coordinate_map.rays
        self._src_geom = source._source_geometry()
        self._device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self._depth = max(1, int(depth))
        self._batch = max(1, int(batch))
        self._streams = [torch.cuda.Stream(device=self._device) for _ in range(self._depth)]
        self._src_bufs: List = [None] * self._depth
        self._dst_bufs: List = [None] * self._depth
        self._pending: List[list] = [[] for _ in range(self._depth)]  # host outputs of the frames a slot holds
        self._rotations: List[list] = [[] for _ in range(self._depth)]  # their rotations (pipelines that take them)
        self._rotated: Optional[bool] = None  # fixed by the first submit
        self._slot = 0
        self.kernel_launches = 0

    @property
    def output_shape(self):
        return (self._rays.out.height, self._rays.out.output_width)

    def _launch(self, slot: int):
        """Remap what slot ``slot`` holds and send it back to the host; -> completion event."""
        torch = self._torch
        outs = self._pending[slot]
        if not outs:
            return None
        n = len(outs)
        stream = self._streams[slot]
        with torch.cuda.device(self._device), torch.cuda.stream(stream):
            src_dev = self._src_bufs[slot]
            if self._dst_bufs[slot] is None:
                oh, ow = self.output_shape
                self._dst_bufs[slot] = torch.empty((self._batch, oh, ow) + tuple(src_dev.shape[3:]), dtype=src_dev.dtype,
                                                   device=self._device)
            dst_dev = self._dst_bufs[slot]
            if self._rotated:
                engine.remap_frames_device(self._rays, self._src_geom, src_dev[:n], self._rotations[slot], dst_dev[:n])
            elif n == 1:  # one frame: the single-frame kernels
                engine.remap_device(self._rays, self._src_geom, src_dev[0], dst_dev[0])
            else:
                engine.remap_device(self._rays, self._src_geom, src_dev[:n], dst_dev[:n])
            self.kernel_launches += 1
            for k, host_out in enumerate(outs):
                host_out.copy_(dst_dev[k], non_blocking=True)
            done = torch.cuda.Event()
            done.record(stream)
        self._pending[slot] = []
        self._rotations[slot] = []
        return done

    def submit(self, host_frame, host_out, rotation=None):
        """Enqueue one frame: host_frame (CPU tensor (H, W, C) of any dtype the remap takes) ->
        host_out (CPU tensor (Ho, Wo, C) of the same dtype), through ``rotation`` (a ``Rotation`` or
        a 3x3 matrix) after the map's rotations when given.  Returns immediately: the completion event of the launch when this
        frame completed a batch, else None."""
        rotated = rotation is not None
        if self._rotated is None:
            self._rotated = rotated
        elif rotated != self._rotated:
            raise ValueError("a FramePipeline takes a rotation with every frame or with none")
        if rotated:
            rotation = engine.frame_matrices([rotation])[0].reshape(3, 3)
        torch = self._torch
        slot = self._slot
        stream = self._streams[slot]
        with torch.cuda.device(self._device), torch.cuda.stream(stream):
            want = (self._batch,) + tuple(host_frame.shape)
            buf = self._src_bufs[slot]
            if buf is None or tuple(buf.shape) != want or buf.dtype != host_frame.dtype:
                engine.check_source(self._src_geom, host_frame)
                self._src_bufs[slot] = torch.empty(want, dtype=host_frame.dtype, device=self._device)
                self._dst_bufs[slot] = None
            self._src_bufs[slot][len(self._pending[slot])].copy_(host_frame, non_blocking=True)
        self._pending[slot].append(host_out)
        if rotated:
            self._rotations[slot].append(rotation)
        if len(self._pending[slot]) < self._batch:
            return None
        self._slot = (slot + 1) % self._depth
        return self._launch(slot)

    def flush(self):
        """Launch a partly filled batch now; -> its completion event (None if nothing was pending)."""
        slot = self._slot
        if not self._pending[slot]:
            return None
        self._slot = (slot + 1) % self._depth
        return self._launch(slot)

    def run(self, host_frames: Sequence, host_outs: Sequence) -> None:
        """Remap every frame of ``host_frames`` into the matching ``host_outs`` and wait."""
        if len(host_frames) != len(host_outs):
            raise ValueError("host_frames and host_outs differ in length")
        for frame, out in zip(host_frames, host_outs):
            self.submit(frame, out)
        self.drain()

    def drain(self) -> None:
        self.flush()
        for s in self._streams:
            s.synchronize()
