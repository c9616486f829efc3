"""make-pano, alter-photo, make-photo.

Same command names, arguments, options and exit behaviour as the reference
(photonbend/scripts/commands/{__init__,make_pano,alter_photo,make_photo}.py):

* output must end in .jpg/.jpeg/.png, otherwise exit 1; an existing output asks
  "File already exists. Overwrite? (y/n)" and exits 0 on "n";
* an unreadable input prints an error and exits 1; an unwritable output likewise;
* fov checks raise ValueError (double image with fov < 180, any fov > 360);
* ``-r/--rotation PITCH YAW ROLL`` (degrees) may be given several times, applied in order;
* ``-s/--size`` sets the height of the output (square, or 2:1 for panoramas / double images);
* the magnitude (pixel radius at which fov/2 is reached) follows the image type: half the width
  minus half a pixel for inscribed and cropped circles, the half-diagonal for full-frame images;
  a double image ignores it.  alter-photo derives the OUTPUT magnitude from the INPUT shape, like
  the reference does (alter_photo.py:142) -- harmless when both have the same shape, and
  reproduced as is otherwise.

A DIRECTORY as INPUT (an extension over the reference: the frames of a video, photos from one
camera) converts every .jpg/.jpeg/.png in it with the same parameters into the OUTPUT directory,
frames sharded over the visible GPUs (photonbend_b200/stream.py); ``--frames-per-launch`` sets how
many frames share a kernel launch.  ``--frame-rotations FILE`` gives every frame a rotation of its
own, applied after the ``-r`` rotations (stabilised or levelled footage, a moving virtual camera):
one line ``<file name> <pitch> <yaw> <roll>`` (degrees) per frame; blank lines and ``#`` comments
are ignored.

Everything between decode and encode runs on the GPU: the source array is uploaded once, the
three-call protocol (get_coordinate_map / rotate_coordinate_map / process_coordinate_map) costs
one kernel launch, and the result is downloaded once.
"""

from __future__ import annotations

import sys
from pathlib import Path
from typing import List, Optional, Tuple

import click
import numpy as np

from photonbend_b200.core import lens as lenses
from photonbend_b200.core.projection import CameraImage, DoubleCameraImage, PanoramaImage
from photonbend_b200.core.rotation import Rotation
from photonbend_b200.utils import image_io, to_radians

CHANNELS = 3
IMAGE_TYPES = ("inscribed", "double", "cropped", "full")
LENS_NAMES = ("equidistant", "equisolid", "orthographic", "rectilinear", "stereographic")

_TYPE_HELP = """

    \b
    The choices are:
    - inscribed: The valid data is on a inscribed circle.
    - double: The valid data is on two inscribed side-by-side circles.
    - cropped: The valid data is on a inscribed circle, top-and-bottom cropped.
    - full: The whole area of the image is valid data.
    """
_DOUBLE_FOV_NOTE = """

    IMPORTANT: FoV for double images are the value for one of the sensors and > 180ª."""
_ROTATION_HELP = """
    The rotation that should be applied to the camera.
    This is a 3-valued parameter in the form <pitch yaw roll>
    """


# ------------------------------------------------------------------------------- shared pieces


def _checked_output(path: Path) -> Path:
    path = Path(path)
    if path.suffix.lower() not in (".jpg", ".jpeg", ".png"):
        print("The desired output image should be a JPG or PNG file.")
        print("Provide an output filename ending in either JPG, JPEG or PNG (case insensitive)")
        print("Exiting!")
        sys.exit(1)
    if path.exists():
        answer = ""
        while answer not in ("y", "n"):
            answer = input("File already exists. Overwrite? (y/n) ")
        if answer == "n":
            print("Exiting!")
            sys.exit(0)
    return path


def _load_pixels(path):
    """uint8 pixels of the input file: a NumPy array (Pillow, the default) or, with
    PHOTONBEND_B200_CODEC=nvjpeg, a CUDA tensor decoded on the device (utils/image_io.py)."""
    try:
        return image_io.open_image(path)
    except IOError:
        print("Error: Input image could not be opened!")
        print("Exiting!")
        sys.exit(1)


def _save_pixels(pixels, path: Path) -> None:
    try:
        image_io.save_image(pixels, path)
    except IOError:
        print("Could not save to the specified location!")
        print("Exiting!")
        sys.exit(1)


def _magnitude(image_type: str, shape: Tuple[int, ...]) -> float:
    """Pixel distance from the centre at which fov / 2 is reached."""
    if len(shape) > 3:
        raise ValueError("Can't calculate magnitude of images with more than 3 dimensions")
    height, width, _ = shape
    if image_type == "double":
        return height / 2 - 0.5
    if image_type == "full":
        return float(np.sqrt((width / 2.0 - 0.5) ** 2 + (height / 2.0 - 0.5) ** 2))
    return width / 2 - 0.5  # inscribed, cropped


def _fov_radians(fov_degrees: float, image_type: str) -> float:
    if image_type == "double" and fov_degrees < 180:
        raise ValueError("The fov of a double image can't be smaller than 180 degrees.")
    if fov_degrees > 360:
        raise ValueError("The fov of an image can't be higher than 360 degrees.")
    return to_radians(fov_degrees)


def _photo(pixels, image_type: str, lens_name: str, fov: float, magnitude: float):
    lens = getattr(lenses, lens_name)()
    if image_type == "double":
        return DoubleCameraImage(pixels, fov, lens, magnitude=magnitude)
    return CameraImage(pixels, fov, lens, magnitude=magnitude)


def _photo_shape(image_type: str, source_shape, size: Optional[int]) -> Tuple[int, int, int]:
    height = source_shape[0] if size is None else size
    return (height, 2 * height if image_type == "double" else height, CHANNELS)


def _remap(source, destination, rotations: List[Tuple[float, float, float]]) -> np.ndarray:
    coordinate_map = destination.get_coordinate_map()
    for pitch, yaw, roll in rotations:
        coordinate_map = Rotation(to_radians(pitch), to_radians(yaw), to_radians(roll)).rotate_coordinate_map(
            coordinate_map)
    return source.process_coordinate_map(coordinate_map)


def _exit_with(message: str) -> None:
    print(message)
    print("Exiting!")
    sys.exit(1)


def _read_frame_rotations(path: Path, files: List[Path]) -> List[Rotation]:
    """The rotation of every frame of ``files`` from a ``--frame-rotations`` file, in frame order;
    exits 1 on a malformed line, a name that is not a frame, a frame listed twice or not at all."""
    try:
        text = Path(path).read_text()
    except (OSError, UnicodeDecodeError):
        _exit_with(f"Error: frame rotations file {path} could not be read!")
    names = {f.name for f in files}
    angles = {}
    for number, line in enumerate(text.splitlines(), 1):
        fields = line.split("#", 1)[0].split()
        if not fields:
            continue
        try:
            if len(fields) != 4:
                raise ValueError
            pitch, yaw, roll = (float(v) for v in fields[1:])
        except ValueError:
            _exit_with(f"Error: {path}:{number}: expected <file name> <pitch> <yaw> <roll>, got {line.strip()!r}")
        name = fields[0]
        if name not in names:
            _exit_with(f"Error: {path}:{number}: {name} is not a frame of the input directory")
        if name in angles:
            _exit_with(f"Error: {path}:{number}: frame {name} is listed twice")
        angles[name] = (pitch, yaw, roll)
    missing = [f.name for f in files if f.name not in angles]
    if missing:
        _exit_with(f"Error: {path} gives no rotation for frame {missing[0]}"
                   + (f" (and {len(missing) - 1} more)" if len(missing) > 1 else ""))
    return [Rotation(to_radians(p), to_radians(y), to_radians(r)) for p, y, r in (angles[f.name] for f in files)]


def _remap_directory(in_dir: Path, out_dir: Path, make_pair, rotations, frames_per_launch: int,
                     frame_rotations: Optional[Path] = None) -> None:
    """Every image of ``in_dir`` through the geometry ``make_pair(first_frame_pixels)`` ->
    (source, destination) into ``out_dir`` (same file names), sharded over the visible GPUs; frame
    k also through its own rotation from the ``frame_rotations`` file when given."""
    from photonbend_b200 import stream

    out_dir = Path(out_dir)
    if out_dir.suffix.lower() in (".jpg", ".jpeg", ".png") or (out_dir.exists() and not out_dir.is_dir()):
        print("The input is a directory of frames: the output must be a directory too.")
        print("Exiting!")
        sys.exit(1)
    files = stream.list_frames(in_dir)
    if not files:
        print("Error: no .jpg / .jpeg / .png frames in the input directory!")
        print("Exiting!")
        sys.exit(1)
    per_frame = None if frame_rotations is None else _read_frame_rotations(frame_rotations, files)
    outs = [out_dir / f.name for f in files]
    if any(o.exists() for o in outs):
        answer = ""
        while answer not in ("y", "n"):
            answer = input("Output frames already exist. Overwrite? (y/n) ")
        if answer == "n":
            print("Exiting!")
            sys.exit(0)
    try:
        out_dir.mkdir(parents=True, exist_ok=True)
    except OSError:
        print("Could not save to the specified location!")
        print("Exiting!")
        sys.exit(1)
    first = _load_pixels(files[0])
    if not isinstance(first, np.ndarray):
        first = first.cpu().numpy()
    source, destination = make_pair(first)
    coordinate_map = destination.get_coordinate_map()
    for pitch, yaw, roll in rotations:
        coordinate_map = Rotation(to_radians(pitch), to_radians(yaw), to_radians(roll)).rotate_coordinate_map(
            coordinate_map)
    try:
        stats = stream.remap_files(source, coordinate_map, files, outs, batch=max(1, frames_per_launch),
                                   frame_rotations=per_frame)
    except IOError:
        print("Could not read or save a frame!")
        print("Exiting!")
        sys.exit(1)
    print(f"{stats['frames']} frames on {stats['gpus']} GPU(s) in {stats['seconds']:.2f} s "
          f"({stats['kernel_launches']} launches, codec {stats['codec']})")


def _frames_option(fn):
    return click.option("--frames-per-launch", required=False, type=click.INT, default=4,
                        help="Directory input only: frames remapped by one kernel launch.")(fn)


def _rotation_option(fn):
    return click.option("-r", "--rotation", required=False, type=click.FLOAT, nargs=3, default=[],
                        help=_ROTATION_HELP, multiple=True)(fn)


def _frame_rotations_option(fn):
    return click.option("--frame-rotations", required=False, default=None,
                        type=click.Path(exists=True, dir_okay=False, path_type=Path),
                        help="Directory input only: a file of '<file name> <pitch> <yaw> <roll>' lines (degrees), "
                             "one rotation per frame, applied after the -r rotations.")(fn)


def _single_image(input_image, frame_rotations) -> bool:
    """True for a single-image INPUT; exits 1 when --frame-rotations was given with one."""
    if Path(input_image).is_dir():
        return False
    if frame_rotations is not None:
        _exit_with("Error: --frame-rotations needs a directory of frames as input.")
    return True


def _size_option(fn):
    return click.option("-s", "--size", required=False, type=click.INT, default=None,
                        help="The vertical size of the destiny image")(fn)


# ------------------------------------------------------------------------------- make-pano


@click.command(name="make-pano")
@click.argument("input_image", type=click.Path(exists=True, path_type=Path))
@click.option("--type", "itype", required=True, type=click.Choice(IMAGE_TYPES),
              help="The type of the input image. " + _TYPE_HELP)
@click.option("--lens", required=True, type=click.Choice(LENS_NAMES),
              help="The lens type that was used on the input photo.")
@click.option("--fov", required=True, type=click.FLOAT,
              help="The lens field of view of the input photo in degrees. " + _DOUBLE_FOV_NOTE)
@_rotation_option
@_size_option
@_frames_option
@_frame_rotations_option
@click.argument("output_image", type=click.Path(exists=False, path_type=Path))
def make_pano(input_image, itype, lens, fov, output_image, rotation, size, frames_per_launch, frame_rotations):
    """Make a panorama out of a photo.

    \b
    INPUT is the path to the source photo (or a directory of frames).
    OUTPUT is the desired path of the destiny panorama (a directory for a directory).
    """
    def pair(pixels):
        source = _photo(pixels, itype, lens, _fov_radians(fov, itype), _magnitude(itype, pixels.shape))
        height = pixels.shape[0] if size is None else size
        return source, PanoramaImage(np.zeros((height, int(height * 2), CHANNELS), np.uint8))

    if not _single_image(input_image, frame_rotations):
        return _remap_directory(input_image, output_image, pair, rotation, frames_per_launch, frame_rotations)
    out = _checked_output(output_image)
    source, destination = pair(_load_pixels(input_image))
    _save_pixels(_remap(source, destination, rotation), out)


# ------------------------------------------------------------------------------- alter-photo


@click.command(name="alter-photo")
@click.argument("input_image", type=click.Path(exists=True, path_type=Path))
@click.option("--itype", required=True, type=click.Choice(IMAGE_TYPES),
              help="The type of the input image. " + _TYPE_HELP)
@click.option("--otype", required=True, type=click.Choice(IMAGE_TYPES),
              help="The type of the output image. " + _TYPE_HELP)
@click.option("--ilens", required=True, type=click.Choice(LENS_NAMES),
              help="The lens type that was used on the input photo.")
@click.option("--olens", required=True, type=click.Choice(LENS_NAMES),
              help="The lens type to use on the output photo.")
@click.option("--ifov", required=True, type=click.FLOAT,
              help="The lens field of view of the input photo in degrees. " + _DOUBLE_FOV_NOTE)
@click.option("--ofov", required=True, type=click.FLOAT,
              help="The lens field of view of the output photo in degrees. " + _DOUBLE_FOV_NOTE)
@_rotation_option
@_size_option
@_frames_option
@_frame_rotations_option
@click.argument("output_image", type=click.Path(exists=False, path_type=Path))
def alter_photo(input_image, itype, ilens, ifov, otype, olens, ofov, output_image, rotation, size, frames_per_launch, frame_rotations):
    """Change the the lens and FoV of a photo.

    \b
    INPUT is the path to the source photo (or a directory of frames).
    OUTPUT is the desired path of the destiny photo (a directory for a directory).
    """
    def pair(pixels):
        source = _photo(pixels, itype, ilens, _fov_radians(ifov, itype), _magnitude(itype, pixels.shape))
        canvas = np.zeros(_photo_shape(otype, pixels.shape, size), np.uint8)
        # output magnitude from the INPUT shape, as the reference does
        return source, _photo(canvas, otype, olens, _fov_radians(ofov, otype), _magnitude(otype, pixels.shape))

    if not _single_image(input_image, frame_rotations):
        return _remap_directory(input_image, output_image, pair, rotation, frames_per_launch, frame_rotations)
    out = _checked_output(output_image)
    source, destination = pair(_load_pixels(input_image))
    _save_pixels(_remap(source, destination, rotation), out)


# ------------------------------------------------------------------------------- make-photo


@click.command(name="make-photo")
@click.argument("input_image", type=click.Path(exists=True, path_type=Path))
@click.option("--type", "otype", required=True, type=click.Choice(IMAGE_TYPES),
              help="The type of the output image. " + _TYPE_HELP)
@click.option("--lens", required=True, type=click.Choice(LENS_NAMES),
              help="The lens type to use on the output photo.")
@click.option("--fov", required=True, type=click.FLOAT,
              help="The lens field of view of the output photo in degrees. " + _DOUBLE_FOV_NOTE)
@_rotation_option
@_size_option
@_frames_option
@_frame_rotations_option
@click.argument("output_image", type=click.Path(exists=False, path_type=Path))
def make_photo(input_image, otype, lens, fov, output_image, rotation, size, frames_per_launch, frame_rotations):
    """Make a photo out of a panorama.

    \b
    INPUT is the path to the source panorama (or a directory of frames).
    OUTPUT is the desired path of the destiny photo (a directory for a directory).
    """
    def pair(pixels):
        shape = _photo_shape(otype, pixels.shape, size)
        return PanoramaImage(pixels), _photo(np.zeros(shape, np.uint8), otype, lens, _fov_radians(fov, otype),
                                             _magnitude(otype, shape))

    if not _single_image(input_image, frame_rotations):
        return _remap_directory(input_image, output_image, pair, rotation, frames_per_launch, frame_rotations)
    out = _checked_output(output_image)
    source, destination = pair(_load_pixels(input_image))
    _save_pixels(_remap(source, destination, rotation), out)


__all__ = ["make_pano", "alter_photo", "make_photo"]
