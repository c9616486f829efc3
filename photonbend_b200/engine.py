"""Host-side engine: geometry descriptors, device buffers (torch is the plumbing for device
memory and streams only) and the calls into libpbremap.so.

Nothing here computes pixels on the CPU; a missing CUDA device or library is an error.
"""

from __future__ import annotations

import ctypes
import threading
from dataclasses import dataclass, field
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _native

_KIND_NAMES = {"camera": _native.KIND_CAMERA, "double": _native.KIND_DOUBLE,
               "equirect": _native.KIND_EQUIRECT}


@dataclass(frozen=True)
class ImageGeometry:
    """One side of a remap, as libpbremap.so wants it (pb_image_desc)."""

    kind: int
    height: int
    width: int
    lens: int = 0
    fov: float = 0.0
    f_distance: float = 0.0
    # LENS_TABLE (a user-defined Lens): float64 samples of the one lens function this side of the
    # remap evaluates, on [0, table_max] (see include/pb_remap.h: pb_image_desc.lens_table)
    table: Optional[np.ndarray] = field(default=None, compare=False)
    table_max: float = 0.0
    table_key: bytes = b""  # digest of ``table``: what two geometries with user lenses are compared by
    # double-fisheye source: blend the two lenses in the image's own dtype instead of refusing
    # anything but uint8 (see check_source).  A property of the calls, not of the descriptor: one
    # cached plan serves both settings.
    keep_dtype: bool = False

    @property
    def output_width(self) -> int:
        # a double image only has 2*(width//2) columns (reference projection.py:389-397)
        return 2 * (self.width // 2) if self.kind == _native.KIND_DOUBLE else self.width

    def fill(self, d: _native.ImageDesc) -> None:
        d.kind, d.lens, d.height, d.width = self.kind, self.lens, self.height, self.width
        d.fov, d.f_distance = float(self.fov), float(self.f_distance)
        if self.lens == _native.LENS_TABLE and self.kind != _native.KIND_EQUIRECT:
            if self.table is None:
                raise ValueError("a LENS_TABLE geometry needs its table")
            d.lens_table = self.table.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # (self keeps it alive)
            d.lens_table_n = int(self.table.size)
            d.lens_table_max = float(self.table_max)

    def table_digest(self) -> bytes:
        if self.table is None:
            return b""
        if self.table_key:
            return self.table_key
        import hashlib

        return hashlib.sha1(self.table.tobytes()).digest()


@dataclass(frozen=True)
class RayPlan:
    """Lazy description of a coordinate map: output geometry + rotation matrices in order."""

    out: ImageGeometry
    rotations: Tuple[Tuple[float, ...], ...] = field(default_factory=tuple)

    def rotated(self, matrix) -> "RayPlan":
        m = tuple(float(v) for v in np.asarray(matrix, dtype=np.float64).reshape(9))
        return RayPlan(self.out, self.rotations + (m,))

    @property
    def shape(self):
        return (self.out.height, self.out.output_width, 3)


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError(
            "photonbend_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback"
        )
    return torch


def _stream_ptr(torch) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


_desc_memo: dict = {}  # (rays, src, channels) -> filled descriptor: a stream of calls through one geometry fills it once


def _remap_desc(rays: RayPlan, src: ImageGeometry, channels: int) -> _native.RemapDesc:
    memo_key = (rays, src, channels)
    hit = _desc_memo.get(memo_key)
    if hit is not None:
        return hit
    d = _build_remap_desc(rays, src, channels)
    if len(_desc_memo) >= 64:
        _desc_memo.pop(next(iter(_desc_memo)))
    _desc_memo[memo_key] = d
    return d


def _build_remap_desc(rays: RayPlan, src: ImageGeometry, channels: int) -> _native.RemapDesc:
    if len(rays.rotations) > _native.PB_MAX_ROTATIONS:
        raise _native.NativeError(_native.PB_ERR_TOO_MANY_ROTATIONS, "too many rotations to fuse")
    d = _native.RemapDesc()
    rays.out.fill(d.out)
    src.fill(d.src)
    d._keep = (rays.out.table, src.table)       # the host tables must outlive the descriptor
    d._tables = rays.out.table_digest() + src.table_digest()
    d.channels = channels
    d.n_rotations = len(rays.rotations)
    for k, m in enumerate(rays.rotations):
        for e in range(9):
            d.rotations[k][e] = m[e]
    return d


# ----------------------------------------------------------------------------- plans


def _desc_key(desc: _native.RemapDesc) -> bytes:
    """Identity of a remap for the plan cache: the descriptor's bytes with the host pointers of
    lens tables replaced by a digest of what they point at."""
    key = getattr(desc, "_key", None)
    if key is not None:
        return key
    tables = getattr(desc, "_tables", b"")
    if not tables:
        key = bytes(desc)
    else:
        clone = _native.RemapDesc.from_buffer_copy(bytes(desc))
        clone.out.lens_table = clone.src.lens_table = None
        key = bytes(clone) + tables
    desc._key = key
    return key


class _PlanCache:
    """pb_plan handles keyed by (device, descriptor bytes): a geometry that is remapped again
    (a video, a batch of photos from one camera) reuses its separable device tables."""

    def __init__(self, capacity: int = 32):
        self._capacity = capacity
        self._plans = {}  # key -> handle (insertion order = LRU order)
        # host threads may share the cache (ctypes releases the GIL inside a call).  A handle that
        # falls out of the cache is destroyed only after the work enqueued with it has finished;
        # a thread that still holds an evicted handle across ``capacity`` other geometries is not
        # supported (launches through one handle are serialised inside the library).
        self._lock = threading.RLock()

    def get(self, lib, desc: _native.RemapDesc, device_index: int, torch) -> ctypes.c_void_p:
        key = (device_index, _desc_key(desc))
        with self._lock:
            handle = self._plans.pop(key, None)
            if handle is None:
                handle = ctypes.c_void_p()
                stream = torch.cuda.current_stream()
                _native.check(lib.pb_plan_create(ctypes.byref(desc), ctypes.c_void_p(stream.cuda_stream),
                                                 ctypes.byref(handle)))
                stream.synchronize()  # once per geometry: the tables may be used from any stream later
                while len(self._plans) >= self._capacity:
                    oldest = next(iter(self._plans))
                    torch.cuda.synchronize(oldest[0])
                    lib.pb_plan_destroy(self._plans.pop(oldest))
            self._plans[key] = handle  # most recently used goes last
            return handle

    def clear(self):
        with self._lock:
            if self._plans:
                lib = _native.load()
                for handle in self._plans.values():
                    lib.pb_plan_destroy(handle)
                self._plans.clear()


_plans = _PlanCache()


def clear_plan_cache() -> None:
    """Destroy every cached pb_plan (frees their device tables)."""
    _plans.clear()


# ----------------------------------------------------------------------------- image plumbing


def is_torch_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


def image_layout(image) -> Tuple[int, int, int, bool]:
    """(height, width, channels, had_channel_axis) of an HWC / HW image."""
    shape = tuple(image.shape)
    if len(shape) == 2:
        return shape[0], shape[1], 1, False
    if len(shape) == 3:
        return shape[0], shape[1], shape[2], True
    raise ValueError(f"expected an (H, W, C) or (H, W) image, got shape {shape}")


# Element types the remap takes, by NumPy / torch name, and their width in bytes.  The remap copies
# a pixel's bytes and converts nothing, so only the width matters (bfloat16: torch tensors only).
ELEM_BYTES = {
    "bool": 1, "int8": 1, "uint8": 1,
    "int16": 2, "uint16": 2, "float16": 2, "bfloat16": 2,
    "int32": 4, "uint32": 4, "float32": 4,
    "int64": 8, "uint64": 8, "float64": 8,
}


def _dtype_name(image) -> str:
    name = str(image.dtype)
    return name[len("torch."):] if name.startswith("torch.") else name


def elem_bytes(image) -> int:
    """Bytes per element of an image the remap takes (see ELEM_BYTES); NotImplementedError naming
    the dtype for anything else (complex, object, structured, non-native byte order ...)."""
    name = _dtype_name(image)
    width = ELEM_BYTES.get(name)
    if width is None or (name == "bfloat16" and not is_torch_tensor(image)):
        raise NotImplementedError(f"images of dtype {name} are not supported: the remap takes bool, int8, uint8, "
                                  "int16, uint16, float16, bfloat16 (torch), int32, uint32, float32, int64, uint64 "
                                  "and float64 images")
    return width


def check_source(src: ImageGeometry, image) -> int:
    """elem_bytes(image), after refusing what a source of geometry ``src`` cannot be: a
    double-fisheye source must be uint8 unless its geometry has ``keep_dtype``.  The reference
    blends its two lenses in float64 and casts the blend to uint8 whatever the input dtype
    (projection.py:459), so a wider source would come back as a uint8 image wrapped mod 256; with
    ``keep_dtype`` the blend is cast to the source's own dtype instead (``typed_blend``)."""
    width = elem_bytes(image)
    name = _dtype_name(image)
    if src.kind == _native.KIND_DOUBLE and name != "uint8" and not src.keep_dtype:
        raise NotImplementedError(
            f"a double-fisheye source must be uint8 (got {name}): the reference blends the two lenses and "
            "casts the blend to uint8 whatever the input dtype, which would wrap other values mod 256; "
            "pass keep_dtype=True to blend in the source's own dtype")
    return width


def typed_blend(src: ImageGeometry, image) -> Optional[int]:
    """The PB_ELEM_* type of ``image`` when a remap from ``src`` blends a double-fisheye source in
    that type (the _typed entry points), else None (uint8, or no blend: the _u8 / _px ones)."""
    name = _dtype_name(image)
    if src.kind == _native.KIND_DOUBLE and src.keep_dtype and name != "uint8":
        return _native.ELEM_TYPES[name]
    return None


def to_device(image):
    """Image of an accepted dtype (numpy / torch CPU / torch CUDA) -> contiguous CUDA tensor of the
    same dtype (async H2D on the current stream; pinned host memory makes it a true async copy)."""
    torch = _torch()
    elem_bytes(image)
    if is_torch_tensor(image):
        t = image
    else:
        arr = np.ascontiguousarray(image)
        if not arr.flags.writeable:  # e.g. np.asarray(PIL image): read-only view, only ever read here
            arr = arr.view()
            try:
                arr.flags.writeable = True
            except ValueError:
                arr = arr.copy()
        t = torch.from_numpy(arr)
    if not t.is_cuda:
        t = t.to("cuda", non_blocking=True)
    return t.contiguous()


def from_device_like(result, like, out=None):
    """Hand a CUDA result back in the flavour of ``like`` (numpy -> numpy, torch CPU -> torch
    CPU, torch CUDA -> the CUDA tensor itself).  ``out`` may be a preallocated (ideally pinned)
    destination of the same flavour."""
    torch = _torch()
    if is_torch_tensor(like) and like.is_cuda:
        if out is not None:
            out.copy_(result)
            return out
        return result
    if out is not None:
        host = out if is_torch_tensor(out) else torch.from_numpy(out)
        host.copy_(result, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out
    host = result.cpu()
    return host if is_torch_tensor(like) else host.numpy()


# ----------------------------------------------------------------------------- calls


def _check_out(out_dev, out_shape, src_dev) -> None:
    if tuple(out_dev.shape) != out_shape or not out_dev.is_contiguous() or out_dev.dtype != src_dev.dtype:
        name = _dtype_name(src_dev)
        raise ValueError(f"out must be a contiguous {name} tensor of shape {out_shape}")


def remap_device(rays: RayPlan, src: ImageGeometry, src_dev, out_dev=None):
    """Fused remap on device tensors.  src_dev: CUDA tensor (H, W[, C]) or a batch (N, H, W, C) of
    an accepted dtype (ELEM_BYTES); returns (and fills) the CUDA output tensor of the same dtype.
    One-byte elements take the uint8 kernels (pb_plan_remap_u8), wider ones pb_plan_remap_px; a
    double-fisheye source blended in its own dtype pb_plan_remap_typed."""
    torch = _torch()
    lib = _native.load()
    e = check_source(src, src_dev)
    batched = src_dev.dim() == 4
    frames = src_dev.shape[0] if batched else 1
    h, w, c, had_c = image_layout(src_dev[0] if batched else src_dev)
    if (h, w) != (src.height, src.width):
        raise ValueError(f"source image is {h}x{w} but its geometry says {src.height}x{src.width}")
    oh, ow = rays.out.height, rays.out.output_width
    out_shape = (oh, ow, c) if had_c else (oh, ow)
    if batched:
        out_shape = (frames,) + out_shape
    if out_dev is None:
        out_dev = torch.empty(out_shape, dtype=src_dev.dtype, device=src_dev.device)
    else:
        _check_out(out_dev, out_shape, src_dev)
    desc = _remap_desc(rays, src, c)
    with torch.cuda.device(src_dev.device):
        plan = _plans.get(lib, desc, src_dev.device.index or 0, torch)
        stream = _stream_ptr(torch)
        src_ptr, dst_ptr = ctypes.c_void_p(src_dev.data_ptr()), ctypes.c_void_p(out_dev.data_ptr())
        src_stride, dst_stride = ctypes.c_int64(h * w * c * e), ctypes.c_int64(oh * ow * c * e)
        typed = typed_blend(src, src_dev)
        if typed is not None:
            _native.check(lib.pb_plan_remap_typed(plan, ctypes.c_int32(typed), src_ptr, src_stride, dst_ptr, dst_stride,
                                                  ctypes.c_int32(frames), stream))
        elif e == 1:  # uint8, int8, bool: the same bytes
            _native.check(lib.pb_plan_remap_u8(plan, src_ptr, src_stride, dst_ptr, dst_stride,
                                               ctypes.c_int32(frames), stream))
        else:
            _native.check(lib.pb_plan_remap_px(plan, ctypes.c_int32(e), src_ptr, src_stride, dst_ptr, dst_stride,
                                               ctypes.c_int32(frames), stream))
    return out_dev


def frame_matrices(matrices) -> np.ndarray:
    """(N, 9) C-contiguous float64 rows of N per-frame rotations: ``Rotation`` objects (their
    ``rotation_matrix``) or 3x3 matrices, or an (N, 3, 3) array."""
    if not isinstance(matrices, np.ndarray):
        matrices = [getattr(m, "rotation_matrix", m) for m in matrices]
    arr = np.ascontiguousarray(np.asarray(matrices, dtype=np.float64))
    if arr.ndim != 3 or arr.shape[1:] != (3, 3):
        raise ValueError(f"frame rotations must be N rotations or an (N, 3, 3) array, got shape {arr.shape}")
    return arr.reshape(-1, 9)


def remap_frames_device(rays: RayPlan, src: ImageGeometry, src_dev, matrices, out_dev=None):
    """Fused remap of a batch in which frame k has a rotation of its own (pb_plan_remap_frames_px):
    frame k equals ``remap_device(rays.rotated(matrices[k]), src, frame k)`` byte for byte.
    ``matrices``: N ``Rotation`` objects or an (N, 3, 3) float64 array.  src_dev: a CUDA batch
    (N, H, W, C) of an accepted dtype (ELEM_BYTES), or ONE image (H, W[, C]) seen through all N
    rotations (source frame stride 0).  Returns (and fills) the (N, Ho, Wo[, C]) CUDA output."""
    torch = _torch()
    lib = _native.load()
    e = check_source(src, src_dev)
    mats = frame_matrices(matrices)
    frames = mats.shape[0]
    batched = src_dev.dim() == 4
    if batched and src_dev.shape[0] != frames:
        raise ValueError(f"{src_dev.shape[0]} source frames but {frames} frame rotations")
    h, w, c, had_c = image_layout(src_dev[0] if batched else src_dev)
    if (h, w) != (src.height, src.width):
        raise ValueError(f"source image is {h}x{w} but its geometry says {src.height}x{src.width}")
    oh, ow = rays.out.height, rays.out.output_width
    out_shape = (frames, oh, ow, c) if had_c else (frames, oh, ow)
    if out_dev is None:
        out_dev = torch.empty(out_shape, dtype=src_dev.dtype, device=src_dev.device)
    else:
        _check_out(out_dev, out_shape, src_dev)
    if len(rays.rotations) + 1 > _native.PB_MAX_ROTATIONS:
        raise _native.NativeError(_native.PB_ERR_TOO_MANY_ROTATIONS, "too many rotations to fuse")
    if frames == 0:
        return out_dev
    desc = _remap_desc(rays, src, c)
    with torch.cuda.device(src_dev.device):
        plan = _plans.get(lib, desc, src_dev.device.index or 0, torch)
        typed = typed_blend(src, src_dev)
        call, elem = (lib.pb_plan_remap_frames_px, e) if typed is None else (lib.pb_plan_remap_frames_typed, typed)
        _native.check(call(
            plan, ctypes.c_int32(elem), mats.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            ctypes.c_void_p(src_dev.data_ptr()), ctypes.c_int64(h * w * c * e if batched else 0),
            ctypes.c_void_p(out_dev.data_ptr()), ctypes.c_int64(oh * ow * c * e), ctypes.c_int32(frames),
            _stream_ptr(torch)))
    return out_dev


def remap_rows_device(rays: RayPlan, src: ImageGeometry, src_dev, row_begin: int, row_end: int, out_dev=None):
    """Output rows [row_begin, row_end) of one frame (pb_plan_remap_rows_u8 / _px): src_dev is the
    WHOLE source image on this device, the result is the band alone, (row_end - row_begin, Wo[, C]),
    of the source's dtype."""
    torch = _torch()
    lib = _native.load()
    e = check_source(src, src_dev)
    if src_dev.dim() == 4:
        raise ValueError("a row band is cut from ONE frame, not from a batch")
    h, w, c, had_c = image_layout(src_dev)
    if (h, w) != (src.height, src.width):
        raise ValueError(f"source image is {h}x{w} but its geometry says {src.height}x{src.width}")
    oh, ow = rays.out.height, rays.out.output_width
    if not 0 <= row_begin <= row_end <= oh:
        raise ValueError(f"rows [{row_begin}, {row_end}) outside an output of {oh} rows")
    out_shape = (row_end - row_begin, ow, c) if had_c else (row_end - row_begin, ow)
    if out_dev is None:
        out_dev = torch.empty(out_shape, dtype=src_dev.dtype, device=src_dev.device)
    else:
        _check_out(out_dev, out_shape, src_dev)
    if row_begin == row_end:
        return out_dev
    desc = _remap_desc(rays, src, c)
    with torch.cuda.device(src_dev.device):
        plan = _plans.get(lib, desc, src_dev.device.index or 0, torch)
        src_ptr, dst_ptr = ctypes.c_void_p(src_dev.data_ptr()), ctypes.c_void_p(out_dev.data_ptr())
        rows = (ctypes.c_int32(row_begin), ctypes.c_int32(row_end), _stream_ptr(torch))
        typed = typed_blend(src, src_dev)
        if typed is not None:
            _native.check(lib.pb_plan_remap_rows_typed(plan, ctypes.c_int32(typed), src_ptr, dst_ptr, *rows))
        elif e == 1:
            _native.check(lib.pb_plan_remap_rows_u8(plan, src_ptr, dst_ptr, *rows))
        else:
            _native.check(lib.pb_plan_remap_rows_px(plan, ctypes.c_int32(e), src_ptr, dst_ptr, *rows))
    return out_dev


def materialize_map_device(rays: RayPlan):
    """float64 CUDA tensor (H, W, 3) of the coordinate map described by ``rays``."""
    torch = _torch()
    lib = _native.load()
    fused = RayPlan(rays.out, rays.rotations[: _native.PB_MAX_ROTATIONS])
    rest = rays.rotations[_native.PB_MAX_ROTATIONS:]
    cmap = torch.empty(rays.shape, dtype=torch.float64, device="cuda")
    desc = _remap_desc(fused, fused.out, 1)
    _native.check(lib.pb_materialize_map_f64(ctypes.byref(desc), ctypes.c_void_p(cmap.data_ptr()),
                                             _stream_ptr(torch)))
    for m in rest:
        cmap = rotate_map_device(cmap, m)
    return cmap


def rotate_map_device(cmap_dev, matrix):
    """Rotation.rotate_coordinate_map on a float64 CUDA map; zeroes the invalid entries of
    ``cmap_dev`` in place like the reference (rotation.py:124-125) and returns the new map."""
    torch = _torch()
    lib = _native.load()
    if cmap_dev.dtype != torch.float64 or cmap_dev.shape[-1] != 3 or not cmap_dev.is_contiguous():
        raise ValueError("coordinate map must be a contiguous float64 (..., 3) tensor")
    out = torch.empty_like(cmap_dev)
    mat = (ctypes.c_double * 9)(*[float(v) for v in np.asarray(matrix, dtype=np.float64).reshape(9)])
    with torch.cuda.device(cmap_dev.device):
        _native.check(lib.pb_rotate_map_f64(mat, ctypes.c_void_p(cmap_dev.data_ptr()),
                                            ctypes.c_void_p(out.data_ptr()),
                                            ctypes.c_int64(cmap_dev.numel() // 3), _stream_ptr(torch)))
    return out


def gather_from_map_device(src: ImageGeometry, cmap_dev, src_dev, out_dev=None):
    """process_coordinate_map on an explicit float64 CUDA map; the result has the source's dtype."""
    torch = _torch()
    lib = _native.load()
    e = check_source(src, src_dev)
    h, w, c, had_c = image_layout(src_dev)
    if (h, w) != (src.height, src.width):
        raise ValueError(f"source image is {h}x{w} but its geometry says {src.height}x{src.width}")
    if cmap_dev.dim() != 3 or cmap_dev.shape[2] != 3 or cmap_dev.dtype != torch.float64:
        raise ValueError("coordinate map must be float64 of shape (H, W, 3)")
    if not cmap_dev.is_contiguous():
        raise ValueError("coordinate map must be contiguous")
    if not (cmap_dev.is_cuda and src_dev.is_cuda) or cmap_dev.device != src_dev.device:
        raise ValueError("coordinate map and source image must live on the same CUDA device")
    if not src_dev.is_contiguous():
        raise ValueError("source image must be contiguous")
    mh, mw = cmap_dev.shape[0], cmap_dev.shape[1]
    out_shape = (mh, mw, c) if had_c else (mh, mw)
    if out_dev is None:
        out_dev = torch.empty(out_shape, dtype=src_dev.dtype, device=src_dev.device)
    elif (tuple(out_dev.shape) != out_shape or not out_dev.is_contiguous() or out_dev.dtype != src_dev.dtype
          or out_dev.device != src_dev.device):
        raise ValueError(f"out must be a contiguous {_dtype_name(src_dev)} tensor of shape {out_shape} on {src_dev.device}")
    d = _native.ImageDesc()
    src.fill(d)
    typed = typed_blend(src, src_dev)
    with torch.cuda.device(src_dev.device):
        if typed is not None:
            _native.check(lib.pb_gather_from_map_typed(
                ctypes.byref(d), ctypes.c_int32(c), ctypes.c_int32(typed), ctypes.c_void_p(cmap_dev.data_ptr()),
                ctypes.c_int32(mh), ctypes.c_int32(mw), ctypes.c_void_p(src_dev.data_ptr()),
                ctypes.c_void_p(out_dev.data_ptr()), _stream_ptr(torch)))
        elif e == 1:
            _native.check(lib.pb_gather_from_map_u8(
                ctypes.byref(d), ctypes.c_int32(c), ctypes.c_void_p(cmap_dev.data_ptr()),
                ctypes.c_int32(mh), ctypes.c_int32(mw), ctypes.c_void_p(src_dev.data_ptr()),
                ctypes.c_void_p(out_dev.data_ptr()), _stream_ptr(torch)))
        else:
            _native.check(lib.pb_gather_from_map_px(
                ctypes.byref(d), ctypes.c_int32(c), ctypes.c_int32(e), ctypes.c_void_p(cmap_dev.data_ptr()),
                ctypes.c_int32(mh), ctypes.c_int32(mw), ctypes.c_void_p(src_dev.data_ptr()),
                ctypes.c_void_p(out_dev.data_ptr()), _stream_ptr(torch)))
    return out_dev


def map_projection_device(cmap_dev, out_dev=None):
    """map_projection (reference projection.py:550-599) of a float64 CUDA map (H, W, 3): uint8 CUDA
    image (H, W, 3); zeroes (lat, lon) of the invalid entries of ``cmap_dev`` in place like the reference."""
    torch = _torch()
    lib = _native.load()
    if cmap_dev.dim() != 3 or cmap_dev.shape[2] != 3 or cmap_dev.dtype != torch.float64 or not cmap_dev.is_cuda:
        raise ValueError("coordinate map must be a float64 CUDA tensor of shape (H, W, 3)")
    if not cmap_dev.is_contiguous():
        raise ValueError("coordinate map must be contiguous")
    mh, mw = cmap_dev.shape[0], cmap_dev.shape[1]
    if out_dev is None:
        out_dev = torch.empty((mh, mw, 3), dtype=torch.uint8, device=cmap_dev.device)
    elif (tuple(out_dev.shape) != (mh, mw, 3) or out_dev.dtype != torch.uint8 or not out_dev.is_contiguous()
          or out_dev.device != cmap_dev.device):
        raise ValueError(f"out must be a contiguous uint8 tensor of shape {(mh, mw, 3)} on {cmap_dev.device}")
    with torch.cuda.device(cmap_dev.device):
        _native.check(lib.pb_map_projection_u8(ctypes.c_void_p(cmap_dev.data_ptr()), ctypes.c_int32(mh), ctypes.c_int32(mw),
                                               ctypes.c_void_p(out_dev.data_ptr()), _stream_ptr(torch)))
    return out_dev
