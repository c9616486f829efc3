"""Per-frame rotations, the parts that need no GPU: pb_plan_remap_frames_px's argument errors (codes and
messages; nothing touches a device) and the --frame-rotations file of the directory commands, whose
every error exits 1 before any device work."""

import ctypes

import numpy as np
import pytest
from click.testing import CliRunner
from PIL import Image

from photonbend_b200 import _native, engine
from photonbend_b200.scripts.main import main

FAKE = ctypes.c_void_p(256)  # never dereferenced: validation fails first
ROTS = (ctypes.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)


def _frames(lib, elem_bytes=1, rots=ROTS, src=FAKE, dst=FAKE, n=1, src_stride=0, dst_stride=0, plan=FAKE):
    return lib.pb_plan_remap_frames_px(plan, elem_bytes, rots, src, src_stride, dst, dst_stride, n, None)


@pytest.mark.parametrize("elem_bytes", [0, 3, 16])
def test_frames_refuses_other_element_widths(elem_bytes):
    lib = _native.load()
    assert _frames(lib, elem_bytes) == _native.PB_ERR_UNSUPPORTED
    assert b"pb_plan_remap_frames_px" in lib.pb_last_error() and b"elem_bytes" in lib.pb_last_error()


def test_frames_refuses_null_pointers():
    lib = _native.load()
    for e in (1, 2, 4, 8):
        for kw in ({"plan": None}, {"rots": None}, {"src": None}, {"dst": None}):
            assert _frames(lib, e, **kw) == _native.PB_ERR_INVALID_ARGUMENT, (e, kw)
            assert b"null" in lib.pb_last_error()


def test_frames_negative_and_zero_frame_counts():
    # (uint8: the checks of wider elements read the plan's source kind, which a fake plan does not have)
    lib = _native.load()
    assert _frames(lib, n=-1) == _native.PB_ERR_INVALID_ARGUMENT
    assert b"negative n_frames" in lib.pb_last_error()
    # nothing to do: the (fake) plan is never looked at
    assert _frames(lib, n=0) == _native.PB_OK


def test_frame_matrices_shapes():
    from photonbend_b200.core.rotation import Rotation

    rots = [Rotation(0.1, 0.2, 0.3), Rotation(-0.4, 0.0, 1.0)]
    mats = engine.frame_matrices(rots)
    assert mats.shape == (2, 9) and mats.dtype == np.float64 and mats.flags.c_contiguous
    assert np.array_equal(mats[1], rots[1].rotation_matrix.reshape(9))
    assert np.array_equal(engine.frame_matrices(np.stack([r.rotation_matrix for r in rots])), mats)
    assert engine.frame_matrices(np.zeros((0, 3, 3))).shape == (0, 9)
    with pytest.raises(ValueError, match="N rotations"):
        engine.frame_matrices(np.zeros((2, 9)))


# ------------------------------------------------------------------------------- --frame-rotations

PANO_ARGS = ["make-pano", "--type", "inscribed", "--lens", "equidistant", "--fov", "200"]


def _frame_dir(tmp_path, names=("a.png", "b.png", "c.png")):
    d = tmp_path / "frames"
    d.mkdir()
    for name in names:
        Image.fromarray(np.zeros((8, 8, 3), np.uint8)).save(d / name)
    return d


@pytest.fixture
def no_device(monkeypatch):
    """Any attempt to reach the GPU (or to read a frame) fails the test."""
    from photonbend_b200 import stream
    from photonbend_b200.scripts import commands

    def refuse(*args, **kwargs):
        raise AssertionError("device work before the --frame-rotations checks")

    monkeypatch.setattr(engine, "_torch", refuse)
    monkeypatch.setattr(stream, "remap_files", refuse)
    monkeypatch.setattr(commands, "_load_pixels", refuse)


@pytest.mark.parametrize("text, message", [
    ("a.png 0 0 0\nb.png 1 2 3\n", "no rotation for frame c.png"),
    ("a.png 0 0 0\nb.png 1 2 3\nc.png 0 0 0\nb.png 0 0 0\n", "listed twice"),
    ("a.png 0 0 0\nb.png 1 2 3\nc.png 0 0 0\nd.png 0 0 0\n", "d.png is not a frame"),
    ("a.png 0 0\nb.png 1 2 3\nc.png 0 0 0\n", "expected <file name> <pitch> <yaw> <roll>"),
    ("a.png 0 0 zero\nb.png 1 2 3\nc.png 0 0 0\n", "expected <file name> <pitch> <yaw> <roll>"),
    ("a.png 0 0 0 0\nb.png 1 2 3\nc.png 0 0 0\n", "expected <file name> <pitch> <yaw> <roll>"),
])
@pytest.mark.parametrize("command", ["make-pano", "alter-photo", "make-photo"])
def test_bad_frame_rotations_exit_1_before_device_work(tmp_path, no_device, text, message, command):
    frames = _frame_dir(tmp_path)
    rot_file = tmp_path / "rotations.txt"
    rot_file.write_text(text)
    args = {
        "make-pano": PANO_ARGS,
        "alter-photo": ["alter-photo", "--itype", "inscribed", "--ilens", "equidistant", "--ifov", "180",
                        "--otype", "inscribed", "--olens", "equisolid", "--ofov", "180"],
        "make-photo": ["make-photo", "--type", "inscribed", "--lens", "equidistant", "--fov", "180"],
    }[command]
    res = CliRunner().invoke(main, args + ["--frame-rotations", str(rot_file), str(frames), str(tmp_path / "out")])
    assert res.exit_code == 1, res.output
    assert message in res.output
    assert not (tmp_path / "out").exists()


def test_frame_rotations_with_a_single_image_exits_1(tmp_path, no_device):
    frames = _frame_dir(tmp_path)
    rot_file = tmp_path / "rotations.txt"
    rot_file.write_text("a.png 0 0 0\n")
    res = CliRunner().invoke(main, PANO_ARGS + ["--frame-rotations", str(rot_file), str(frames / "a.png"),
                                                str(tmp_path / "out.png")])
    assert res.exit_code == 1, res.output
    assert "needs a directory of frames" in res.output
    assert not (tmp_path / "out.png").exists()


def test_frame_rotations_file_parses_comments_and_blank_lines(tmp_path):
    from photonbend_b200.core.rotation import Rotation
    from photonbend_b200.scripts import commands
    from photonbend_b200.utils import to_radians

    frames = _frame_dir(tmp_path)
    rot_file = tmp_path / "rotations.txt"
    rot_file.write_text("# name pitch yaw roll\n\nc.png  -1.5\t2 3   # last\n  a.png 0 0 0\nb.png 10 -20 30.25\n")
    files = sorted(frames.iterdir())
    got = commands._read_frame_rotations(rot_file, files)
    want = [(0, 0, 0), (10, -20, 30.25), (-1.5, 2, 3)]
    assert len(got) == 3
    for rot, (p, y, r) in zip(got, want):
        ref = Rotation(to_radians(p), to_radians(y), to_radians(r)).rotation_matrix
        assert np.array_equal(rot.rotation_matrix, ref)
