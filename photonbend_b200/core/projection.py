"""Projection images -- same surface as the reference's photonbend/core/projection.py
(ProjectionImage :40-66, CameraImage :69-274, DoubleCameraImage :277-462, PanoramaImage
:465-547), with the per-pixel work done by libpbremap.so on a B200.

    destination.get_coordinate_map()            -> lazy CoordinateMap (no kernel, no memory)
    Rotation(...).rotate_coordinate_map(map)    -> lazy CoordinateMap with one more matrix
    source.process_coordinate_map(map)          -> ONE fused kernel: ray -> rotate -> index -> sample

Images are HWC (or HW) and may be NumPy arrays, torch CPU tensors (pin them for truly
asynchronous copies) or torch CUDA tensors (device resident: no copies at all, and
``(N, H, W, C)`` batches of frames that share the geometry are remapped by one launch).  Their
elements may be bool, int8, uint8, int16, uint16, float16, bfloat16 (torch), int32, uint32,
float32, int64, uint64 or float64: like the reference's fancy indexing, every output pixel is a
bit-for-bit copy of the source pixel its index picks (0 where there is none).  A double-fisheye
source blends its two lenses: the reference casts that blend to uint8, so a source of another
dtype is refused unless it is made with ``keep_dtype=True``, which casts the blend to the source's
own dtype instead.  The result comes back in the same dtype and flavour as the source image.
"""

from __future__ import annotations

from typing import Optional, Protocol, Union
from abc import abstractmethod

import numpy as np

from photonbend_b200 import _native, engine
from photonbend_b200.core.coordinate_map import CoordinateMap
from photonbend_b200.core.lens import Lens, lens_id, lens_table


class ProjectionImage(Protocol):
    """Protocol shared by every projection image."""

    image: np.ndarray

    @abstractmethod
    def get_coordinate_map(self):
        """The coordinate map (latitude, longitude, invalid) of this image's pixel grid."""
        ...

    @abstractmethod
    def process_coordinate_map(self, coordinate_map):
        """A new image: this image sampled along the rays of ``coordinate_map``."""
        ...


def _frame_shape(image):
    """(height, width) of an image or of the frames of an (N, H, W, C) device batch."""
    shape = tuple(image.shape)
    if len(shape) == 4:
        return shape[1], shape[2]
    return shape[0], shape[1]


def _custom_lens_table(image, lens: int, role: str, height: int, width: int):
    """(samples, range) of the lens function a user-defined Lens needs on this side of a remap --
    as a source the forward function on [0, pi] (latitudes), as an output the reverse function on
    [0, largest pixel radius in focal units] -- cached on the image object; (None, 0) for the
    built-in models."""
    if lens != _native.LENS_TABLE:
        return None, 0.0, b""
    cache = image.__dict__.setdefault("_lens_tables", {})
    key = (role, height, width, float(image.f_distance))
    if key not in cache:
        import hashlib

        if role == "source":
            x_max = float(np.pi)
            fn = image.forward_lens
        else:
            x_max = float(np.hypot((width - 1) / 2.0, (height - 1) / 2.0) / image.f_distance) * (1.0 + 1e-9) + 1e-12
            fn = image.reverse_lens
        table = lens_table(fn, x_max)
        cache[key] = (table, x_max, hashlib.sha1(table.tobytes()).digest())
    return cache[key]


class _DeviceSampler:
    """process_coordinate_map shared by the three image formats."""

    image = None

    def _source_geometry(self) -> engine.ImageGeometry:
        raise NotImplementedError

    def _output_geometry(self) -> engine.ImageGeometry:
        raise NotImplementedError

    def get_coordinate_map(self) -> CoordinateMap:
        """Coordinate map of this image's pixel grid, as a lazy CoordinateMap (it behaves like
        the float64 (H, W, 3) array of (latitude, longitude, invalid) when looked at)."""
        return CoordinateMap(engine.RayPlan(self._output_geometry()))

    def process_coordinate_map(self, coordinate_map, out=None):
        """Sample this image along ``coordinate_map`` and return the new image (same dtype).

        Args:
            coordinate_map: a CoordinateMap from ``get_coordinate_map`` /
                ``rotate_coordinate_map`` (fused path), or an explicit float64 (H, W, 3) map as
                an ndarray or CUDA tensor (explicit-map path).
            out: optional preallocated destination of the same flavour as ``self.image``
                (a pinned torch CPU tensor makes the device-to-host copy asynchronous).
        """
        src_geom = self._source_geometry()
        engine.check_source(src_geom, self.image)  # before any device work
        src_dev = engine.to_device(self.image)

        if isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy \
                and len(coordinate_map.rays.rotations) <= _native.PB_MAX_ROTATIONS:
            rays = coordinate_map.rays
            if src_geom.kind == _native.KIND_EQUIRECT:
                coordinate_map._mark_invalid_zeroed()  # projection.py:533-536
            out_dev = out if (out is not None and engine.is_torch_tensor(out) and out.is_cuda) else None
            result = engine.remap_device(rays, src_geom, src_dev, out_dev)
            if out_dev is not None:
                return out_dev
            return engine.from_device_like(result, self.image, out)

        # explicit map: ndarray, CUDA tensor, or a CoordinateMap that was looked at / edited
        if src_dev.dim() == 4:
            raise ValueError("a batch of frames needs a lazy coordinate map")
        torch = engine._torch()
        host_map = None
        if isinstance(coordinate_map, CoordinateMap):
            if coordinate_map.is_lazy:  # more rotations than one launch fuses
                map_dev = engine.materialize_map_device(coordinate_map.rays)
            else:
                host_map = coordinate_map.materialize()
        elif engine.is_torch_tensor(coordinate_map):
            map_dev = coordinate_map
            if not map_dev.is_cuda:
                raise ValueError("a torch coordinate map must live on the CUDA device")
        else:
            host_map = coordinate_map
        if host_map is not None:
            if not isinstance(host_map, np.ndarray) or host_map.ndim != 3 or host_map.shape[2] != 3:
                raise ValueError("coordinate map must be a float64 array of shape (H, W, 3)")
            map_dev = torch.from_numpy(np.ascontiguousarray(host_map, dtype=np.float64)).cuda()
        result = engine.gather_from_map_device(src_geom, map_dev, src_dev)
        if host_map is not None and src_geom.kind == _native.KIND_EQUIRECT:
            host_map[host_map[:, :, 2] != 0.0, :2] = 0  # side effect of projection.py:533-536
        return engine.from_device_like(result, self.image, out)


class CameraImage(_DeviceSampler):
    """A photo taken through a lens: maps pixels to (latitude, longitude) and back.

    Attributes:
        image: the image, shape (height, width, channels), of any dtype the remap takes.
        fov (float): field of view in radians.
        forward_lens / reverse_lens: the lens functions.
        magnitude (float): distance in pixels from the image centre at which ``fov / 2`` is
            reached (height / 2 by default, i.e. an inscribed circle).
        f_distance (float): focal distance in pixels.
    """

    def __init__(self, image_arr, fov: float, lens: Lens, magnitude: Union[None, float] = None):
        self.image = image_arr
        self.fov = fov
        self.forward_lens = lens.forward_function
        self.reverse_lens = lens.reverse_function
        height = _frame_shape(image_arr)[0]
        self.magnitude: float = (height / 2.0) if (magnitude is None) else magnitude
        self.f_distance = self._compute_f_distance()

    def _compute_f_distance(self) -> float:
        """Pixels per focal unit: the lens projects ``fov / 2`` at ``forward(fov / 2)`` focal
        units, and that has to land ``magnitude`` pixels from the centre.  (The rectilinear
        forward function raises ValueError here for fov / 2 > 89 degrees.)"""
        return self.magnitude / self.forward_lens(self.fov / 2)

    def _geometry(self, role: str) -> engine.ImageGeometry:
        height, width = _frame_shape(self.image)
        lens = lens_id(self.forward_lens, self.reverse_lens)
        table, table_max, table_key = _custom_lens_table(self, lens, role, height, width)
        return engine.ImageGeometry(
            kind=_native.KIND_CAMERA, height=height, width=width, lens=lens,
            fov=float(self.fov), f_distance=float(self.f_distance), table=table, table_max=table_max,
            table_key=table_key)

    def _source_geometry(self):
        return self._geometry("source")

    def _output_geometry(self):
        return self._geometry("output")


class DoubleCameraImage(_DeviceSampler):
    """A 360-degree camera frame: two opposite fisheye sensors stored side by side.

    Attributes:
        image: the image, shape (height, width, channels); each half is width // 2 wide.
        sensor_fov (float): field of view of ONE sensor in radians (> pi for full coverage).
        lens (Lens), forward_lens, reverse_lens: the lens model of both sensors.
        magnitude (float): always height / 2 (a ``magnitude=`` keyword is accepted and ignored).
        f_distance (float): focal distance in pixels.
        keep_dtype (bool): how the two lenses' samples are blended.  False (the default, the
            reference's behaviour): into uint8, and only a uint8 image is accepted (the reference
            casts the float64 blend to uint8 whatever the input dtype, which would wrap wider
            values mod 256).  True: into the image's own dtype -- any dtype the remap takes --
            as ``(left.astype(float64) * w_left + right.astype(float64) * w_right).astype(dtype)``
            with NumPy's casts (bfloat16: torch's); a uint8 image gives the default's bytes.
    """

    def __init__(self, image_arr, sensor_fov: float, lens: Lens, keep_dtype: bool = False, **kwargs):
        self.image = image_arr
        self.keep_dtype = bool(keep_dtype)
        self.sensor_fov = sensor_fov
        self.lens = lens
        self.forward_lens = lens.forward_function
        self.reverse_lens = lens.reverse_function
        self.magnitude = _frame_shape(image_arr)[0] / 2.0
        self.f_distance = self._compute_f_distance()

    def _compute_f_distance(self) -> float:
        return self.magnitude / self.forward_lens(self.sensor_fov / 2)

    def _geometry(self, role: str) -> engine.ImageGeometry:
        height, width = _frame_shape(self.image)
        lens = lens_id(self.forward_lens, self.reverse_lens)
        table, table_max, table_key = _custom_lens_table(self, lens, role, height, width // 2)
        return engine.ImageGeometry(
            kind=_native.KIND_DOUBLE, height=height, width=width, lens=lens,
            fov=float(self.sensor_fov), f_distance=float(self.f_distance), table=table, table_max=table_max,
            table_key=table_key, keep_dtype=self.keep_dtype and role == "source")

    def _source_geometry(self):
        return self._geometry("source")

    def _output_geometry(self):
        return self._geometry("output")


class PanoramaImage(_DeviceSampler):
    """An equirectangular panorama (width = 2 x height).

    Attributes:
        image: the image, shape (height, width, channels), of any dtype the remap takes.
    """

    def __init__(self, image_arr) -> None:
        self.image = image_arr

    def _geometry(self) -> engine.ImageGeometry:
        height, width = _frame_shape(self.image)
        return engine.ImageGeometry(kind=_native.KIND_EQUIRECT, height=height, width=width)

    _source_geometry = _geometry
    _output_geometry = _geometry


def map_projection(coordinate_map) -> np.ndarray:
    """Visualise a coordinate map as an RGB image: latitude -> red (stretched over the range it
    takes on the valid pixels), longitude -> green, invalid -> blue (the reference's debug helper,
    projection.py:550-599).  Runs on the GPU (pb_map_projection_u8): a lazy CoordinateMap is
    materialised on the device and never visits the host; an ndarray is uploaded.  Like the
    reference, (lat, lon) of the invalid entries of an ndarray argument are zeroed in place."""
    torch = engine._torch()
    if isinstance(coordinate_map, CoordinateMap) and coordinate_map.is_lazy:
        dev = engine.materialize_map_device(coordinate_map.rays)
        coordinate_map._mark_invalid_zeroed()
    elif engine.is_torch_tensor(coordinate_map) and coordinate_map.is_cuda:
        dev = coordinate_map  # zeroed in place by the kernel
    else:
        arr = coordinate_map.materialize() if isinstance(coordinate_map, CoordinateMap) else coordinate_map
        if not (isinstance(arr, np.ndarray) and arr.dtype == np.float64 and arr.ndim == 3 and arr.shape[2] == 3):
            raise ValueError("coordinate map must be float64 of shape (H, W, 3)")
        dev = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
        arr[arr[:, :, 2] != 0.0, :2] = 0  # projection.py:566 writes through a view of the caller's map
    if not bool((dev[:, :, 2] == 0).any()):
        # numpy.min of an empty selection (projection.py:570)
        raise ValueError("zero-size array to reduction operation minimum which has no identity")
    return engine.map_projection_device(dev).cpu().numpy()
