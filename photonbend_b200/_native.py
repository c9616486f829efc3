"""ctypes binding of libpbremap.so (include/pb_remap.h).

There is no CPU fallback: if the library is missing and cannot be built, or a call fails,
this module raises.
"""

from __future__ import annotations

import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libpbremap.so")

PB_MAX_ROTATIONS = 16

KIND_CAMERA, KIND_DOUBLE, KIND_EQUIRECT = 0, 1, 2
(LENS_EQUIDISTANT, LENS_EQUISOLID, LENS_ORTHOGRAPHIC, LENS_STEREOGRAPHIC, LENS_RECTILINEAR,
 LENS_THOBY, LENS_TABLE) = range(7)
PB_ABI_VERSION = 2

PB_OK = 0
PB_ERR_INVALID_ARGUMENT = 1
PB_ERR_UNSUPPORTED = 2
PB_ERR_CUDA = 3
PB_ERR_TOO_MANY_ROTATIONS = 4

# element types of the _typed entry points (PB_ELEM_*), by NumPy / torch dtype name
ELEM_TYPES = {
    "uint8": 0, "int8": 1, "bool": 2, "uint16": 3, "int16": 4, "float16": 5, "uint32": 6, "int32": 7,
    "float32": 8, "uint64": 9, "int64": 10, "float64": 11, "bfloat16": 12,
}

# kernel families of pb_debug_launch_counts, in the order of the PB_LAUNCH_* enum
LAUNCH_FAMILIES = ("direct", "direct32", "generic", "tiled", "tiled_sep", "two_lens", "boxes1", "boxes2", "sep1",
                   "chunk", "wide", "gather", "plan", "map", "diagnostic", "frames", "blend")

# every symbol include/pb_remap.h declares
EXPORTS = (
    "pb_version",
    "pb_last_error",
    "pb_kernel_launches",
    "pb_debug_launch_counts",
    "pb_output_width",
    "pb_remap_u8",
    "pb_plan_create",
    "pb_plan_remap_u8",
    "pb_plan_remap_rows_u8",
    "pb_plan_destroy",
    "pb_materialize_map_f64",
    "pb_rotate_map_f64",
    "pb_gather_from_map_u8",
    "pb_map_projection_u8",
    "pb_debug_fast32_stats",
    "pb_debug_plan_fast32",
    "pb_debug_plan_boxes",
    "pb_debug_plan_stage",
    "pb_plan_remap_px",
    "pb_plan_remap_rows_px",
    "pb_gather_from_map_px",
    "pb_plan_remap_frames_px",
    "pb_plan_remap_typed",
    "pb_plan_remap_rows_typed",
    "pb_plan_remap_frames_typed",
    "pb_gather_from_map_typed",
)


class ImageDesc(ctypes.Structure):
    _fields_ = [
        ("kind", ctypes.c_int32),
        ("lens", ctypes.c_int32),
        ("height", ctypes.c_int32),
        ("width", ctypes.c_int32),
        ("fov", ctypes.c_double),
        ("f_distance", ctypes.c_double),
        ("lens_table", ctypes.POINTER(ctypes.c_double)),  # LENS_TABLE: host samples of the lens function
        ("lens_table_n", ctypes.c_int32),
        ("reserved_", ctypes.c_int32),
        ("lens_table_max", ctypes.c_double),
    ]


class RemapDesc(ctypes.Structure):
    _fields_ = [
        ("out", ImageDesc),
        ("src", ImageDesc),
        ("channels", ctypes.c_int32),
        ("n_rotations", ctypes.c_int32),
        ("rotations", (ctypes.c_double * 9) * PB_MAX_ROTATIONS),
    ]


class NativeError(RuntimeError):
    """A libpbremap.so call returned a PB_ERR_* code."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libpbremap error {code}: {message}")
        self.code = code


_lib = None


def load():
    """Load (building once with nvcc if the .so is absent) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PB_REMAP_LIB") or LIB_PATH  # override: A/B runs of experiment builds
    if path == LIB_PATH and not os.path.exists(LIB_PATH):
        from . import build as _build  # raises if nvcc is unavailable or compilation fails

        _build.build()
    lib = ctypes.CDLL(path)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.pb_version.restype = ctypes.c_int
    lib.pb_version.argtypes = []
    lib.pb_last_error.restype = ctypes.c_char_p
    lib.pb_last_error.argtypes = []
    lib.pb_kernel_launches.restype = ctypes.c_int64
    lib.pb_kernel_launches.argtypes = []
    lib.pb_debug_launch_counts.restype = ctypes.c_int
    lib.pb_debug_launch_counts.argtypes = [ctypes.POINTER(ctypes.c_int64), i32]
    lib.pb_output_width.restype = i32
    lib.pb_output_width.argtypes = [ctypes.POINTER(ImageDesc)]
    lib.pb_remap_u8.restype = ctypes.c_int
    lib.pb_remap_u8.argtypes = [ctypes.POINTER(RemapDesc), vp, i64, vp, i64, i32, vp]
    lib.pb_plan_create.restype = ctypes.c_int
    lib.pb_plan_create.argtypes = [ctypes.POINTER(RemapDesc), vp, ctypes.POINTER(vp)]
    lib.pb_plan_remap_u8.restype = ctypes.c_int
    lib.pb_plan_remap_u8.argtypes = [vp, vp, i64, vp, i64, i32, vp]
    lib.pb_plan_remap_rows_u8.restype = ctypes.c_int
    lib.pb_plan_remap_rows_u8.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.pb_plan_destroy.restype = None
    lib.pb_plan_destroy.argtypes = [vp]
    lib.pb_materialize_map_f64.restype = ctypes.c_int
    lib.pb_materialize_map_f64.argtypes = [ctypes.POINTER(RemapDesc), vp, vp]
    lib.pb_rotate_map_f64.restype = ctypes.c_int
    lib.pb_rotate_map_f64.argtypes = [ctypes.POINTER(ctypes.c_double), vp, vp, i64, vp]
    lib.pb_gather_from_map_u8.restype = ctypes.c_int
    lib.pb_gather_from_map_u8.argtypes = [ctypes.POINTER(ImageDesc), i32, vp, i32, i32, vp, vp, vp]
    lib.pb_map_projection_u8.restype = ctypes.c_int
    lib.pb_map_projection_u8.argtypes = [vp, i32, i32, vp, vp]
    lib.pb_debug_fast32_stats.restype = ctypes.c_int
    lib.pb_debug_fast32_stats.argtypes = [ctypes.POINTER(RemapDesc), ctypes.POINTER(ctypes.c_double), vp]
    lib.pb_debug_plan_fast32.restype = ctypes.c_int
    lib.pb_debug_plan_fast32.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    lib.pb_debug_plan_boxes.restype = ctypes.c_int
    lib.pb_debug_plan_boxes.argtypes = [vp, ctypes.POINTER(ctypes.c_int32), ctypes.c_int64, ctypes.POINTER(ctypes.c_int32)]
    lib.pb_debug_plan_stage.restype = ctypes.c_int
    lib.pb_debug_plan_stage.argtypes = [vp, ctypes.POINTER(ctypes.c_int32)]
    lib.pb_plan_remap_px.restype = ctypes.c_int
    lib.pb_plan_remap_px.argtypes = [vp, i32, vp, i64, vp, i64, i32, vp]
    lib.pb_plan_remap_rows_px.restype = ctypes.c_int
    lib.pb_plan_remap_rows_px.argtypes = [vp, i32, vp, vp, i32, i32, vp]
    lib.pb_gather_from_map_px.restype = ctypes.c_int
    lib.pb_gather_from_map_px.argtypes = [ctypes.POINTER(ImageDesc), i32, i32, vp, i32, i32, vp, vp, vp]
    lib.pb_plan_remap_frames_px.restype = ctypes.c_int
    lib.pb_plan_remap_frames_px.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_double), vp, i64, vp, i64, i32, vp]
    lib.pb_plan_remap_typed.restype = ctypes.c_int
    lib.pb_plan_remap_typed.argtypes = [vp, i32, vp, i64, vp, i64, i32, vp]
    lib.pb_plan_remap_rows_typed.restype = ctypes.c_int
    lib.pb_plan_remap_rows_typed.argtypes = [vp, i32, vp, vp, i32, i32, vp]
    lib.pb_plan_remap_frames_typed.restype = ctypes.c_int
    lib.pb_plan_remap_frames_typed.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_double), vp, i64, vp, i64, i32, vp]
    lib.pb_gather_from_map_typed.restype = ctypes.c_int
    lib.pb_gather_from_map_typed.argtypes = [ctypes.POINTER(ImageDesc), i32, i32, vp, i32, i32, vp, vp, vp]
    _lib = lib
    return lib


def launch_counts() -> dict:
    """Kernels launched per family (LAUNCH_FAMILIES) since the process started."""
    lib = load()
    counts = (ctypes.c_int64 * len(LAUNCH_FAMILIES))()
    n = lib.pb_debug_launch_counts(counts, len(LAUNCH_FAMILIES))
    if n != len(LAUNCH_FAMILIES):
        raise RuntimeError(f"libpbremap counts {n} kernel families, this binding knows {len(LAUNCH_FAMILIES)}")
    return dict(zip(LAUNCH_FAMILIES, counts))


def check(code: int) -> None:
    if code != PB_OK:
        msg = load().pb_last_error()
        raise NativeError(code, msg.decode("utf-8", "replace") if msg else "")
