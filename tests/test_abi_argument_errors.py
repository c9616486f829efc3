"""Argument errors of the remap entry points, row by row: the exact code and pb_last_error() text
for each input, including inputs that break two rules at once, so that the order of the checks is
pinned.  Nothing here reaches a device: every row fails (or returns PB_OK for an empty call) before
the library touches one.

The plan entry points read three int fields of a plan before they launch anything: the source kind,
the output height and the device the plan was made on.  A buffer whose every 32-bit word is K stands
in for a plan with source kind K, K output rows and device K.  K = -1 matches no device, so a call
through it fails at the device check on any machine; K = 1 (a double-fisheye source) is only used in
rows that fail before that check.
"""

import ctypes

import pytest

from photonbend_b200 import _native as N

INVALID, UNSUPPORTED, TOO_MANY = N.PB_ERR_INVALID_ARGUMENT, N.PB_ERR_UNSUPPORTED, N.PB_ERR_TOO_MANY_ROTATIONS

FAKE = 256  # never dereferenced; aligned for every element width
ODD, TWO = 257, 258  # aligned to 1 byte, to 2 bytes

_plans = {k: (ctypes.c_int32 * (1 << 14))(*([k] * (1 << 14))) for k in (-1, 1)}
OTHER_DEVICE = ctypes.addressof(_plans[-1])  # camera-like source, H = -1: every row range is outside
DOUBLE_SRC = ctypes.addressof(_plans[1])  # double-fisheye source, H = 1


def image(kind=N.KIND_CAMERA, height=8, width=16, lens=N.LENS_EQUIDISTANT, **kw):
    d = N.ImageDesc()
    d.kind, d.height, d.width, d.lens, d.fov, d.f_distance = kind, height, width, lens, 3.0, 4.0
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def desc(out=None, src=None, channels=3, n_rotations=0):
    d = N.RemapDesc()
    d.out = out if out is not None else image(N.KIND_EQUIRECT)
    d.src = src if src is not None else image()
    d.channels, d.n_rotations = channels, n_rotations
    return d


def remap(d=desc(), src=FAKE, sfs=0, dst=FAKE, dfs=0, n=1):
    return "pb_remap_u8", (ctypes.byref(d) if d is not None else None, src, sfs, dst, dfs, n, None)


def plan_u8(plan=OTHER_DEVICE, src=FAKE, sfs=0, dst=FAKE, dfs=0, n=1):
    return "pb_plan_remap_u8", (plan, src, sfs, dst, dfs, n, None)


def plan_px(e, plan=OTHER_DEVICE, src=FAKE, sfs=0, dst=FAKE, dfs=0, n=1):
    return "pb_plan_remap_px", (plan, e, src, sfs, dst, dfs, n, None)


def rows_u8(rb, re, plan=OTHER_DEVICE, src=FAKE, dst=FAKE):
    return "pb_plan_remap_rows_u8", (plan, src, dst, rb, re, None)


def rows_px(e, rb, re, plan=OTHER_DEVICE, src=FAKE, dst=FAKE):
    return "pb_plan_remap_rows_px", (plan, e, src, dst, rb, re, None)


def gather_u8(sd=image(), ch=3, m=FAKE, mh=4, mw=4, src=FAKE, dst=FAKE):
    return "pb_gather_from_map_u8", (ctypes.byref(sd) if sd is not None else None, ch, m, mh, mw, src, dst, None)


def gather_px(e, sd=image(), ch=3, m=FAKE, mh=4, mw=4, src=FAKE, dst=FAKE):
    return "pb_gather_from_map_px", (ctypes.byref(sd) if sd is not None else None, ch, e, m, mh, mw, src, dst, None)


BIG = 2**31 - 1
TABLE_MSG = "PB_LENS_TABLE needs lens_table (>= 2 samples) and lens_table_max > 0"
TABLE = ctypes.cast(FAKE, ctypes.POINTER(ctypes.c_double))  # never dereferenced: the checks come first
DOUBLE_MSG = ("a double-fisheye source blends its two lenses into uint8 (projection.py:459); "
              "only elem_bytes == 1 is supported for it")
ALIGN_MSG = "pointer or stride not a multiple of elem_bytes"
SIZE_MSG = "source larger than 32767 rows x 65535 columns"

# (call, code, message); message None: PB_OK.  A row whose id ends in "fwd" is a _px call with
# elem_bytes == 1 that fails after the width and null checks: its message may name either the _px
# entry point or the matching _u8 one.
CASES = {
    # pb_remap_u8
    "remap-null-src": (remap(src=None), INVALID, "pb_remap_u8: null pointer"),
    "remap-null-dst+desc": (remap(d=None, dst=None), INVALID, "pb_remap_u8: null pointer"),
    "remap-null-desc+neg-frames": (remap(d=None, n=-1), INVALID, "pb_remap_u8: null descriptor"),
    "remap-out-kind+src-kind": (remap(desc(image(5), image(-1))), INVALID, "out: unknown image kind"),
    "remap-out-size+src-kind": (remap(desc(image(N.KIND_EQUIRECT, height=0), image(7))), INVALID,
                                "out: height and width must be positive"),
    "remap-out-pixels": (remap(desc(image(N.KIND_EQUIRECT, height=65536, width=32768))), UNSUPPORTED,
                         "out: more than 2^31 pixels"),
    "remap-src-kind+channels": (remap(desc(src=image(3), channels=0)), INVALID, "src: unknown image kind"),
    "remap-src-lens+size": (remap(desc(src=image(lens=7, height=40000))), INVALID, "src: unknown lens"),
    "remap-src-table": (remap(desc(src=image(lens=N.LENS_TABLE))), INVALID, "src: " + TABLE_MSG),
    "remap-src-table-2^24+1": (remap(desc(src=image(lens=N.LENS_TABLE, lens_table=TABLE, lens_table_n=(1 << 24) + 1,
                                                    lens_table_max=3.0))), INVALID, "src: " + TABLE_MSG),
    "remap-out-table-inf-max": (remap(desc(out=image(lens=N.LENS_TABLE, lens_table=TABLE, lens_table_n=2,
                                                     lens_table_max=float("inf"))), n=0), INVALID, "out: " + TABLE_MSG),
    "remap-src-table-nan-max": (remap(desc(src=image(lens=N.LENS_TABLE, lens_table=TABLE, lens_table_n=17,
                                                     lens_table_max=float("nan")))), INVALID, "src: " + TABLE_MSG),
    "remap-src-table-zero-max": (remap(desc(src=image(N.KIND_DOUBLE, lens=N.LENS_TABLE, lens_table=TABLE,
                                                      lens_table_n=17, lens_table_max=0.0))), INVALID, "src: " + TABLE_MSG),
    "remap-out-table-neg-max": (remap(desc(out=image(lens=N.LENS_TABLE, lens_table=TABLE, lens_table_n=1 << 24,
                                                     lens_table_max=-1.0))), INVALID, "out: " + TABLE_MSG),
    "gather-table-2^24+1": (gather_u8(sd=image(lens=N.LENS_TABLE, lens_table=TABLE, lens_table_n=(1 << 24) + 1,
                                               lens_table_max=3.0)), INVALID, "src: " + TABLE_MSG),
    "remap-src-double-width": (remap(desc(src=image(N.KIND_DOUBLE, width=1))), INVALID,
                               "src: a double image needs width >= 2"),
    "remap-equirect-ignores-lens": (remap(desc(src=image(N.KIND_EQUIRECT, lens=99)), n=0), N.PB_OK, None),
    "remap-src-rows+channels": (remap(desc(src=image(height=32768), channels=5)), UNSUPPORTED,
                                "pb_remap_u8: " + SIZE_MSG),
    "remap-src-cols": (remap(desc(src=image(N.KIND_EQUIRECT, height=2, width=65536))), UNSUPPORTED,
                       "pb_remap_u8: " + SIZE_MSG),
    "remap-channels+rotations": (remap(desc(channels=5, n_rotations=-1)), UNSUPPORTED,
                                 "pb_remap_u8: channels must be 1..4"),
    "remap-neg-rotations+frames": (remap(desc(n_rotations=-1), n=-1), INVALID, "pb_remap_u8: negative n_rotations"),
    "remap-many-rotations+frames": (remap(desc(n_rotations=N.PB_MAX_ROTATIONS + 1), n=-1), TOO_MANY,
                                    "pb_remap_u8: more than PB_MAX_ROTATIONS rotations"),
    "remap-neg-frames": (remap(n=-1), INVALID, "pb_remap_u8: negative n_frames"),
    "remap-zero-frames": (remap(n=0), N.PB_OK, None),
    # pb_plan_remap_u8
    "plan-null-plan": (plan_u8(plan=None), INVALID, "pb_plan_remap_u8: null pointer"),
    "plan-null-dst+frames": (plan_u8(dst=None, n=-1), INVALID, "pb_plan_remap_u8: null pointer"),
    "plan-neg-frames": (plan_u8(n=-1), INVALID, "pb_plan_remap_u8: negative n_frames"),
    "plan-zero-frames": (plan_u8(n=0), N.PB_OK, None),
    "plan-zero-frames-double": (plan_u8(plan=DOUBLE_SRC, n=0), N.PB_OK, None),
    "plan-device": (plan_u8(), INVALID, "pb_plan_remap_u8: plan belongs to another device"),
    # pb_plan_remap_px
    "px-width+null": (plan_px(3, plan=None), UNSUPPORTED, "pb_plan_remap_px: elem_bytes must be 1, 2, 4 or 8 (got 3)"),
    "px-width-neg": (plan_px(-2), UNSUPPORTED, "pb_plan_remap_px: elem_bytes must be 1, 2, 4 or 8 (got -2)"),
    "px-null+double": (plan_px(2, plan=DOUBLE_SRC, src=None), INVALID, "pb_plan_remap_px: null pointer"),
    "px-null-e1": (plan_px(1, dst=None, n=-1), INVALID, "pb_plan_remap_px: null pointer"),
    "px-double+align": (plan_px(4, plan=DOUBLE_SRC, src=ODD, n=-1), UNSUPPORTED, "pb_plan_remap_px: " + DOUBLE_MSG),
    "px-double-e8": (plan_px(8, plan=DOUBLE_SRC, n=0), UNSUPPORTED, "pb_plan_remap_px: " + DOUBLE_MSG),
    "px-align-src+frames": (plan_px(2, src=ODD, n=-1), INVALID, "pb_plan_remap_px: " + ALIGN_MSG),
    "px-align-src-stride": (plan_px(4, sfs=6, n=0), INVALID, "pb_plan_remap_px: " + ALIGN_MSG),
    "px-align-dst": (plan_px(4, dst=TWO, n=0), INVALID, "pb_plan_remap_px: " + ALIGN_MSG),
    "px-align-dst-stride": (plan_px(8, dfs=4, n=0), INVALID, "pb_plan_remap_px: " + ALIGN_MSG),
    "px-aligned-e2": (plan_px(2, src=TWO, dst=TWO, sfs=2, dfs=6, n=0), N.PB_OK, None),
    "px-neg-frames": (plan_px(8, n=-1), INVALID, "pb_plan_remap_px: negative n_frames"),
    "px-zero-frames": (plan_px(2, n=0), N.PB_OK, None),
    "px-device": (plan_px(4), INVALID, "pb_plan_remap_px: plan belongs to another device"),
    "px-e1-skips-wide-checks": (plan_px(1, plan=DOUBLE_SRC, src=ODD, sfs=3, n=0), N.PB_OK, None),
    "px-neg-frames-fwd": (plan_px(1, plan=DOUBLE_SRC, src=ODD, n=-1), INVALID, "pb_plan_remap_px: negative n_frames"),
    "px-device-fwd": (plan_px(1, src=ODD), INVALID, "pb_plan_remap_px: plan belongs to another device"),
    # pb_plan_remap_rows_u8
    "rows-null-src+rows": (rows_u8(-1, 0, src=None), INVALID, "pb_plan_remap_rows_u8: null pointer"),
    "rows-neg-begin": (rows_u8(-1, 0, plan=DOUBLE_SRC), INVALID, "pb_plan_remap_rows_u8: rows outside the output image"),
    "rows-end-past-h": (rows_u8(0, 2, plan=DOUBLE_SRC), INVALID, "pb_plan_remap_rows_u8: rows outside the output image"),
    "rows-begin-past-end": (rows_u8(1, 0, plan=DOUBLE_SRC), INVALID,
                            "pb_plan_remap_rows_u8: rows outside the output image"),
    "rows-empty": (rows_u8(1, 1, plan=DOUBLE_SRC), N.PB_OK, None),
    "rows-outside-before-device": (rows_u8(0, 0), INVALID, "pb_plan_remap_rows_u8: rows outside the output image"),
    # pb_plan_remap_rows_px
    "rowspx-width+null": (rows_px(0, 0, 0, plan=None), UNSUPPORTED,
                          "pb_plan_remap_rows_px: elem_bytes must be 1, 2, 4 or 8 (got 0)"),
    "rowspx-width-16": (rows_px(16, 0, 0), UNSUPPORTED, "pb_plan_remap_rows_px: elem_bytes must be 1, 2, 4 or 8 (got 16)"),
    "rowspx-null+double": (rows_px(2, 0, 0, plan=DOUBLE_SRC, dst=None), INVALID, "pb_plan_remap_rows_px: null pointer"),
    "rowspx-double+align+rows": (rows_px(2, -1, 0, plan=DOUBLE_SRC, dst=ODD), UNSUPPORTED,
                                 "pb_plan_remap_rows_px: " + DOUBLE_MSG),
    "rowspx-align-src+rows": (rows_px(8, 0, 0, src=TWO + 2), INVALID, "pb_plan_remap_rows_px: " + ALIGN_MSG),
    "rowspx-align-dst+rows": (rows_px(2, -1, 0, dst=ODD), INVALID, "pb_plan_remap_rows_px: " + ALIGN_MSG),
    "rowspx-rows": (rows_px(4, 0, 0, src=TWO + 2, dst=TWO + 6), INVALID,
                    "pb_plan_remap_rows_px: rows outside the output image"),
    "rowspx-e1-skips-wide-checks": (rows_px(1, 1, 1, plan=DOUBLE_SRC, src=ODD), N.PB_OK, None),
    "rowspx-rows-fwd": (rows_px(1, 0, 2, plan=DOUBLE_SRC, dst=ODD), INVALID,
                        "pb_plan_remap_rows_px: rows outside the output image"),
    # pb_gather_from_map_u8
    "gather-null-map+desc": (gather_u8(sd=image(9), m=None), INVALID, "pb_gather_from_map_u8: null pointer"),
    "gather-null-desc": (gather_u8(sd=None), INVALID, "pb_gather_from_map_u8: null pointer"),
    "gather-kind+size": (gather_u8(sd=image(9, height=40000)), INVALID, "src: unknown image kind"),
    "gather-lens+channels": (gather_u8(sd=image(lens=-1), ch=0), INVALID, "src: unknown lens"),
    "gather-table": (gather_u8(sd=image(N.KIND_DOUBLE, lens=N.LENS_TABLE, lens_table_n=1)), INVALID,
                     "src: " + TABLE_MSG),
    "gather-size+channels": (gather_u8(sd=image(width=70000), ch=5), UNSUPPORTED, "pb_gather_from_map_u8: " + SIZE_MSG),
    "gather-channels+map": (gather_u8(ch=5, mh=-1), UNSUPPORTED, "pb_gather_from_map_u8: channels must be 1..4"),
    "gather-neg-map": (gather_u8(mw=-4), INVALID, "pb_gather_from_map_u8: negative map size"),
    "gather-empty-map": (gather_u8(mh=0, mw=BIG), N.PB_OK, None),
    "gather-map-too-large": (gather_u8(mh=BIG, mw=BIG), UNSUPPORTED, "pb_gather_from_map_u8: map too large"),
    # pb_gather_from_map_px
    "gatherpx-width+null": (gather_px(5, sd=None), UNSUPPORTED,
                            "pb_gather_from_map_px: elem_bytes must be 1, 2, 4 or 8 (got 5)"),
    "gatherpx-null+kind": (gather_px(2, sd=image(9), src=None), INVALID, "pb_gather_from_map_px: null pointer"),
    "gatherpx-kind+double-align": (gather_px(2, sd=image(-3), src=ODD), INVALID, "src: unknown image kind"),
    "gatherpx-table+align": (gather_px(4, sd=image(lens=N.LENS_TABLE), dst=ODD), INVALID, "src: " + TABLE_MSG),
    "gatherpx-double+align": (gather_px(8, sd=image(N.KIND_DOUBLE), src=ODD, ch=0), UNSUPPORTED,
                              "pb_gather_from_map_px: " + DOUBLE_MSG),
    "gatherpx-align-src+size": (gather_px(4, sd=image(height=40000), src=TWO), INVALID,
                                "pb_gather_from_map_px: " + ALIGN_MSG),
    "gatherpx-align-dst+channels": (gather_px(2, dst=ODD, ch=9), INVALID, "pb_gather_from_map_px: " + ALIGN_MSG),
    "gatherpx-size+channels": (gather_px(2, sd=image(N.KIND_EQUIRECT, height=32768, width=2), ch=9), UNSUPPORTED,
                               "pb_gather_from_map_px: " + SIZE_MSG),
    "gatherpx-channels+map": (gather_px(8, ch=0, mw=-1), UNSUPPORTED, "pb_gather_from_map_px: channels must be 1..4"),
    "gatherpx-neg-map": (gather_px(4, mh=-1), INVALID, "pb_gather_from_map_px: negative map size"),
    "gatherpx-empty-map": (gather_px(2, mh=BIG, mw=0), N.PB_OK, None),
    "gatherpx-map-too-large": (gather_px(8, mh=BIG, mw=BIG), UNSUPPORTED, "pb_gather_from_map_px: map too large"),
    "gatherpx-e1-double": (gather_px(1, sd=image(N.KIND_DOUBLE), src=ODD, dst=ODD, mh=0), N.PB_OK, None),
    "gatherpx-e1-kind": (gather_px(1, sd=image(4)), INVALID, "src: unknown image kind"),
    "gatherpx-size-fwd": (gather_px(1, sd=image(height=32768)), UNSUPPORTED, "pb_gather_from_map_px: " + SIZE_MSG),
    "gatherpx-channels-fwd": (gather_px(1, ch=0, src=ODD), UNSUPPORTED, "pb_gather_from_map_px: channels must be 1..4"),
    "gatherpx-neg-map-fwd": (gather_px(1, mh=-1), INVALID, "pb_gather_from_map_px: negative map size"),
    "gatherpx-map-too-large-fwd": (gather_px(1, mh=BIG, mw=BIG), UNSUPPORTED, "pb_gather_from_map_px: map too large"),
}


@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_argument_error(case):
    (fn, args), code, want = CASES[case]
    lib = N.load()
    assert getattr(lib, fn)(*args) == code
    if want is None:
        return
    got = lib.pb_last_error().decode()
    if case.endswith("-fwd"):
        # the _px call hands elem_bytes == 1 to the uint8 body, which may report under the _u8 name
        assert got in (want, want.replace("_px:", "_u8:", 1))
    else:
        assert got == want
