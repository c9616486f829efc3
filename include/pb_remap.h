/*
 * pb_remap.h -- C ABI of libpbremap.so, the B200 (sm_100a) implementation of photonbend's
 * per-pixel remap path.
 *
 * The reference (wmoreirae/photonbend) is pure Python + NumPy and has no FFI of its own; the
 * boundary these entry points replace is its ProjectionImage protocol
 * (photonbend/core/__init__.py:51-92, photonbend/core/projection.py:40-66):
 *
 *     map = dst.get_coordinate_map()                      projection.py:147, 341, 487
 *     map = Rotation(p, y, r).rotate_coordinate_map(map)  rotation.py:102-176   (0..n times)
 *     out = src.process_coordinate_map(map)               projection.py:197, 408, 515
 *
 * pb_remap_u8 fuses the three calls into one kernel launch; the other three entry points are
 * the same protocol with the float64 coordinate map materialised in device memory, for
 * callers that inspect or edit the map between the calls.
 *
 * Conventions
 *  - every pointer marked "device" is a CUDA device pointer on the CURRENT device; the caller
 *    allocates and owns every buffer; the library allocates nothing that outlives a call, except
 *    the small tables owned by a pb_plan (see below);
 *  - source images may have at most 32767 rows and 65535 columns;
 *  - images are HWC, tightly packed (row pitch = width * channels elements): uint8 for the _u8
 *    entry points; the _px entry points take elements of 1, 2, 4 or 8 bytes of any type (a pixel
 *    is copied as bytes, never converted), except from a double-fisheye source, whose blend is
 *    uint8 arithmetic; the _typed entry points take a PB_ELEM_* type and blend a double-fisheye
 *    source in that type;
 *  - coordinate maps are float64 (H, W, 3) = (latitude, longitude, invalid != 0), tightly packed
 *    (photonbend/core/__init__.py:42-49);
 *  - all work is enqueued on `stream` (a cudaStream_t, NULL = the default stream) and the call
 *    returns without synchronising;
 *  - every function returns PB_OK (0) or a PB_ERR_* code; pb_last_error() gives the message of
 *    the last failure on the calling thread.  Nothing throws or aborts across the ABI;
 *  - host-side parameter derivation stays with the caller exactly as the reference does it:
 *    f_distance = magnitude / lens_forward(fov / 2) (projection.py:123-144, 318-339) and the
 *    row-major 3x3 matrices Rotation.rotation_matrix (rotation.py:27-62, 100), so that these
 *    constants are bit-identical to the reference's.
 */
#ifndef PB_REMAP_H
#define PB_REMAP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_ABI_VERSION 2

/* image formats: projection.py CameraImage :69, DoubleCameraImage :277, PanoramaImage :465 */
enum { PB_KIND_CAMERA = 0, PB_KIND_DOUBLE = 1, PB_KIND_EQUIRECT = 2 };

/* lens models: lens.py:341-401 */
enum {
    PB_LENS_EQUIDISTANT = 0,
    PB_LENS_EQUISOLID = 1,
    PB_LENS_ORTHOGRAPHIC = 2,
    PB_LENS_STEREOGRAPHIC = 3,
    PB_LENS_RECTILINEAR = 4,
    PB_LENS_THOBY = 5,
    /* a user-defined lens (lens.py:48-64 lets Lens wrap any pair of callables): the function the
     * kernel needs is handed over as a table of samples, see pb_image_desc.lens_table */
    PB_LENS_TABLE = 6
};

enum {
    PB_OK = 0,
    PB_ERR_INVALID_ARGUMENT = 1,
    PB_ERR_UNSUPPORTED = 2,
    PB_ERR_CUDA = 3,
    PB_ERR_TOO_MANY_ROTATIONS = 4
};

#define PB_MAX_ROTATIONS 16

/* One side (output or source) of a remap. */
typedef struct pb_image_desc {
    int32_t kind;      /* PB_KIND_* */
    int32_t lens;      /* PB_LENS_*; ignored for PB_KIND_EQUIRECT */
    int32_t height;    /* pixels */
    int32_t width;     /* pixels (a double image holds two width/2 halves side by side) */
    double fov;        /* radians: full field of view (camera) or per-sensor fov (double) */
    double f_distance; /* pixels per focal unit = magnitude / lens_forward(fov / 2) */
    /* PB_LENS_TABLE only (otherwise NULL / 0): 2 <= lens_table_n <= 2^24 float64 samples in HOST
     * memory of the one lens function this side of the remap evaluates (lens_table_max finite and
     * > 0, else PB_ERR_INVALID_ARGUMENT), at x_k = k * lens_table_max /
     * (lens_table_n - 1): as `out`, the lens's reverse function (radius in focal units ->
     * latitude); as `src`, its forward function (latitude -> radius in focal units).  The kernel
     * interpolates linearly and clamps x to [0, lens_table_max].  Copied during the call (plans
     * keep a device copy): the caller may free it afterwards.  Results follow the user's callables
     * to the interpolation error, not bit for bit -- the only lens kind for which that holds. */
    const double *lens_table;
    int32_t lens_table_n;
    int32_t reserved_;
    double lens_table_max;
} pb_image_desc;

/* A whole remap: output geometry, rotations applied in order, source geometry. */
typedef struct pb_remap_desc {
    pb_image_desc out;
    pb_image_desc src;
    int32_t channels;    /* 1..4 interleaved channels (uint8, or the element width of a _px call) */
    int32_t n_rotations; /* 0..PB_MAX_ROTATIONS */
    double rotations[PB_MAX_ROTATIONS][9]; /* row-major Rotation.rotation_matrix, in order */
} pb_remap_desc;

int pb_version(void);
const char *pb_last_error(void);

/* Kernels this library has launched in this process so far (every grid counts once; a batch
 * through a double-fisheye source is two grids, one per tile class).  For benchmarks that have to
 * state how many of their own kernels ran inside a timed region. */
int64_t pb_kernel_launches(void);

/* Kernel families of pb_debug_launch_counts: which kernel a launch ran. */
enum {
    PB_LAUNCH_DIRECT = 0,     /* remap_direct_kernel: one frame, float64 tiers per pixel */
    PB_LAUNCH_DIRECT32 = 1,   /* remap_direct32_kernel: one frame, FP32-first tier */
    PB_LAUNCH_GENERIC = 2,    /* remap_generic_kernel: any layout, alignment or stride */
    PB_LAUNCH_TILED = 3,      /* remap_tiled_kernel, generic rays (MODE 0) */
    PB_LAUNCH_TILED_SEP = 4,  /* remap_tiled_kernel, separable tables (MODE 1), every tile class */
    PB_LAUNCH_TWO_LENS = 5,   /* remap_two_lens_kernel */
    PB_LAUNCH_BOXES1 = 6,     /* remap_boxes_kernel, one-lens tiles */
    PB_LAUNCH_BOXES2 = 7,     /* remap_boxes_kernel, two-lens and blend-band tiles */
    PB_LAUNCH_SEP1 = 8,       /* remap_sep1_kernel: one frame, separable */
    PB_LAUNCH_CHUNK = 9,      /* remap_chunk_kernel */
    PB_LAUNCH_WIDE = 10,      /* remap_wide_kernel: elements wider than a byte */
    PB_LAUNCH_GATHER = 11,    /* gather_from_map_kernel: explicit maps */
    PB_LAUNCH_PLAN = 12,      /* plan-time kernels: tables, footprints, boxes, census, calibration */
    PB_LAUNCH_MAP = 13,       /* coordinate-map kernels: materialise, rotate, map_projection */
    PB_LAUNCH_DIAGNOSTIC = 14, /* pb_debug_fast32_stats */
    PB_LAUNCH_FRAMES = 15,    /* remap_frames_kernel: a rotation per frame (pb_plan_remap_frames_px) */
    PB_LAUNCH_BLEND = 16,     /* remap_blend_kernel: a double-fisheye batch blended in its own type */
    PB_LAUNCH_FAMILIES = 17
};

/* Element types of the _typed entry points (NumPy's names; bfloat16 as torch's). */
enum {
    PB_ELEM_UINT8 = 0,
    PB_ELEM_INT8 = 1,
    PB_ELEM_BOOL = 2,
    PB_ELEM_UINT16 = 3,
    PB_ELEM_INT16 = 4,
    PB_ELEM_FLOAT16 = 5,
    PB_ELEM_UINT32 = 6,
    PB_ELEM_INT32 = 7,
    PB_ELEM_FLOAT32 = 8,
    PB_ELEM_UINT64 = 9,
    PB_ELEM_INT64 = 10,
    PB_ELEM_FLOAT64 = 11,
    PB_ELEM_BFLOAT16 = 12
};

/* Kernels launched per family since the process started, for tests that must know which kernel
 * a call ran.  Fills counts[0 .. min(capacity, PB_LAUNCH_FAMILIES)) (nothing when counts is NULL)
 * and returns PB_LAUNCH_FAMILIES.  The families add up to pb_kernel_launches(). */
int pb_debug_launch_counts(int64_t *counts, int32_t capacity);

/* Width of the image a geometry produces: 2*(width/2) for PB_KIND_DOUBLE (projection.py:389-397),
 * width otherwise. */
int32_t pb_output_width(const pb_image_desc *out);

/*
 * Fused remap of n_frames frames that share one geometry:
 *   dst[k] = src_format.process_coordinate_map(rotate*(out_format.get_coordinate_map()))  on src[k]
 * src: device, n_frames images of src.height x src.width x channels, frame k at src + k*src_frame_stride
 * dst: device, n_frames images of out.height x pb_output_width(out) x channels, likewise.
 */
int pb_remap_u8(const pb_remap_desc *desc, const uint8_t *src, int64_t src_frame_stride,
                uint8_t *dst, int64_t dst_frame_stride, int32_t n_frames, void *stream);

/*
 * Plans.  A plan is one validated geometry together with everything derived from it: the host
 * constants and, for an un-rotated equirect output (the video case, BASELINE config 5), small
 * separable device tables (cos/sin of each column's longitude, lens radius of each row's
 * latitude; 16*W + 32*H bytes) that the kernel would otherwise rebuild per call.  pb_remap_u8 is
 * pb_plan_create + pb_plan_remap_u8 + pb_plan_destroy with the tables in a transient
 * stream-ordered allocation.  The tables are the only device memory the library ever owns; they
 * live on the device that was current at pb_plan_create and die with pb_plan_destroy.
 * pb_plan_create enqueues the table kernel on `stream`; use the plan on that stream or after it.
 */
typedef struct pb_plan pb_plan;
int pb_plan_create(const pb_remap_desc *desc, void *stream, pb_plan **plan);
int pb_plan_remap_u8(const pb_plan *plan, const uint8_t *src, int64_t src_frame_stride, uint8_t *dst,
                     int64_t dst_frame_stride, int32_t n_frames, void *stream);
/*
 * Output rows [row_begin, row_end) of ONE frame: dst_band (device) holds (row_end - row_begin) x
 * pb_output_width(out) x channels bytes, i.e. the band alone.  This is how a single large frame is
 * sharded over the GPUs of a box by output-row bands: every GPU holds the whole source and
 * produces its own band, no exchange (the reference's protocol works on any row slice of the
 * coordinate map the same way: photonbend/core/projection.py:197-245 takes any (h, w, 3) map).
 * Bands that start on a multiple of 64 rows take the TMA-staged kernels.
 */
int pb_plan_remap_rows_u8(const pb_plan *plan, const uint8_t *src, uint8_t *dst_band,
                          int32_t row_begin, int32_t row_end, void *stream);
/*
 * Like the _u8 entry points, for pixels of desc->channels elements of elem_bytes (1, 2, 4 or 8)
 * bytes each (uint16, float16, bfloat16, float32, int32, float64 ...); strides in bytes.  Every
 * output pixel is a bit-for-bit copy of the source pixel the reference's index picks, or all-zero
 * bytes.  elem_bytes == 1 is exactly the _u8 call.  src / dst aligned to elem_bytes.  One plan
 * serves every element width: the width is a property of the call.  Errors, before any device
 * work: elem_bytes not in {1, 2, 4, 8} -> PB_ERR_UNSUPPORTED; a double-fisheye source with
 * elem_bytes > 1 -> PB_ERR_UNSUPPORTED (its blend is uint8 arithmetic, projection.py:459); a null
 * pointer, or a pointer / stride not a multiple of elem_bytes -> PB_ERR_INVALID_ARGUMENT.  A batch
 * is one kernel launch whatever n_frames is.
 */
int pb_plan_remap_px(const pb_plan *plan, int32_t elem_bytes, const void *src, int64_t src_frame_stride,
                     void *dst, int64_t dst_frame_stride, int32_t n_frames, void *stream);
int pb_plan_remap_rows_px(const pb_plan *plan, int32_t elem_bytes, const void *src, void *dst_band,
                          int32_t row_begin, int32_t row_end, void *stream);
/*
 * A batch whose frames each have a rotation of their own (stabilised or levelled 360-degree video, a
 * virtual camera moving through a panorama): frame k of the batch is remapped as if desc->rotations
 * had frame_rotations[k] (row-major 3x3, HOST memory, n_frames x 9 doubles, read during the call)
 * appended as its last rotation -- byte-identical to pb_plan_remap_px through a plan of that
 * descriptor.  Strides, element widths and their errors as pb_plan_remap_px (elem_bytes == 1 is
 * uint8); a source stride of 0 gives n_frames views of one image.  desc->n_rotations + 1 >
 * PB_MAX_ROTATIONS -> PB_ERR_TOO_MANY_ROTATIONS before any device work.  A frame whose matrix is not
 * orthonormal or not finite takes the exact float64 chain, as a plan of it would.  Kernel launches
 * only (one per 128 frames): no allocation, no synchronisation, so the call can be captured into a
 * CUDA graph.
 */
int pb_plan_remap_frames_px(const pb_plan *plan, int32_t elem_bytes, const double *frame_rotations,
                            const void *src, int64_t src_frame_stride, void *dst, int64_t dst_frame_stride,
                            int32_t n_frames, void *stream);
/*
 * The _px entry points with an element TYPE (PB_ELEM_*) in place of a width.  For a camera or
 * equirect source they are the _px call with the type's width.  For a double-fisheye source the
 * two lenses are blended in the source's own type: every output element is
 *     (double)left * w_left + (double)right * w_right          (products rounded, no FMA)
 * cast to the element type as NumPy's astype does on x86-64 (bfloat16: as torch's cast, through
 * float32), with a missing lens sample counting as 0 and pixels outside the output's fov 0 -- the
 * reference's blend (projection.py:459) with its final cast to uint8 replaced.  PB_ELEM_UINT8 is
 * exactly the uint8 path.  A batch through a double-fisheye source is one launch of
 * remap_blend_kernel whatever n_frames is.  Errors, before any device work: an unknown type ->
 * PB_ERR_UNSUPPORTED; a null pointer, or a pointer / stride not a multiple of the type's width ->
 * PB_ERR_INVALID_ARGUMENT; the rest as the _px call.
 */
int pb_plan_remap_typed(const pb_plan *plan, int32_t elem_type, const void *src, int64_t src_frame_stride, void *dst,
                        int64_t dst_frame_stride, int32_t n_frames, void *stream);
int pb_plan_remap_rows_typed(const pb_plan *plan, int32_t elem_type, const void *src, void *dst_band,
                             int32_t row_begin, int32_t row_end, void *stream);
int pb_plan_remap_frames_typed(const pb_plan *plan, int32_t elem_type, const double *frame_rotations,
                               const void *src, int64_t src_frame_stride, void *dst, int64_t dst_frame_stride,
                               int32_t n_frames, void *stream);
void pb_plan_destroy(pb_plan *plan);

/*
 * get_coordinate_map() followed by desc->n_rotations rotate_coordinate_map() calls, written to
 * map (device, float64 out.height x pb_output_width(out) x 3).  desc->src is ignored.
 */
int pb_materialize_map_f64(const pb_remap_desc *desc, double *map, void *stream);

/*
 * Rotation.rotate_coordinate_map on an explicit map of n_pixels entries (rotation.py:102-176):
 * map_out = rotated map; like the reference, the invalid entries of map_in are zeroed in place.
 * map_in and map_out are device pointers and may not alias.
 */
int pb_rotate_map_f64(const double matrix[9], double *map_in, double *map_out, int64_t n_pixels,
                      void *stream);

/*
 * process_coordinate_map on an explicit map (device, float64 map_height x map_width x 3):
 * dst (device, map_height x map_width x channels) = src image sampled through the map.
 * Like the reference's PanoramaImage.process_coordinate_map (projection.py:533-536), an
 * equirect source zeroes the invalid entries of map in place.
 */
int pb_gather_from_map_u8(const pb_image_desc *src_desc, int32_t channels, double *map,
                          int32_t map_height, int32_t map_width, const uint8_t *src, uint8_t *dst,
                          void *stream);
/* The same for elements of elem_bytes (1, 2, 4 or 8) bytes, with the errors of pb_plan_remap_px. */
int pb_gather_from_map_px(const pb_image_desc *src_desc, int32_t channels, int32_t elem_bytes, double *map,
                          int32_t map_height, int32_t map_width, const void *src, void *dst, void *stream);
/* The same for elements of type elem_type (PB_ELEM_*), as pb_plan_remap_typed. */
int pb_gather_from_map_typed(const pb_image_desc *src_desc, int32_t channels, int32_t elem_type, double *map,
                             int32_t map_height, int32_t map_width, const void *src, void *dst, void *stream);

/*
 * map_projection (projection.py:550-599) on an explicit map (device, float64 map_height x
 * map_width x 3): dst (device, map_height x map_width x 3 uint8) = (latitude stretched over the
 * range it takes on the valid pixels, longitude * 255 / 2 pi, 255 where invalid), each rounded half
 * to even and cast like numpy's astype(uint8).  Like the reference it zeroes (lat, lon) of the
 * invalid entries of map in place.  A map without a valid pixel makes the reference raise
 * (numpy.min of an empty array); callers check that themselves -- here the red channel is then 0.
 */
int pb_map_projection_u8(double *map, int32_t map_height, int32_t map_width, uint8_t *dst, void *stream);

/*
 * Diagnostics of the FP32-first tier of the per-pixel chain (csrc/pb_fast32.cuh), over every output
 * pixel of a geometry, synchronous: stats[0..1] = largest |float - double| / (2^-24 * error shape)
 * of a source coordinate along x / y (the calibration of the tier's error bound K), stats[2] =
 * pixels, stats[3] = pixels the tier left undecided (they take the float64 tiers), stats[4] = pixels
 * it decided DIFFERENTLY from the float64 tiers (must be 0), stats[5] = pixels whose fov / no-pixel
 * status float and double evaluations disagree on (must be 0).  No reference counterpart: the
 * reference computes in float64 throughout (projection.py:37,46,57).
 */
int pb_debug_fast32_stats(const pb_remap_desc *desc, double stats[6], void *stream);

/*
 * The FP32-first tier as calibrated for one plan: pb_plan_create measures the largest
 * |float - double| / (2^-24 * error shape) over the plan's own output pixels (out[1]; -1 when the
 * plan resolves through tables and needs no tier) and bounds the tier's error with
 * K = max(1.5, 1.25 * that + 0.25) (out[0]; 0 when the tier is off) instead of the K = 16 that holds for
 * every geometry.  No reference counterpart.
 */
int pb_debug_plan_fast32(const pb_plan *plan, double out[2]);

/*
 * The per-box extents a plan of a separable double-fisheye geometry stages for batches (csrc/pb_boxes.cuh),
 * synchronous: dims = {tiles_y, tiles_x, boxes per (tile, slot)}, all 0 when the plan has no such table.
 * With table non-null (capacity >= tiles_y * tiles_x * 2 * boxes * 4 int32) it receives one entry per
 * (tile in raster order, slot: left / right lens, box): {first staged byte of the box's rows, width in
 * 16-byte units (0: nothing staged; -1 in every entry of a tile that is not described), byte offset of
 * the box inside a frame group, first source row of its 16}.  No reference counterpart.
 */
int pb_debug_plan_boxes(const pb_plan *plan, int32_t *table, int64_t capacity, int32_t dims[3]);

/*
 * The staging sizes a plan picked from its footprint census at pb_plan_create, and those its batches
 * launch with: out = {stage-buffer bytes of remap_tiled_kernel, widest staged row in 16-byte units
 * (the plan's widest tensor map), stage buffers of a batch through remap_tiled_kernel, stage-buffer
 * bytes of the single-frame kernel for a camera source, the same for a double-fisheye source's
 * two-lens tiles (or every tile), the same for its one-lens tiles, frame-group ring bytes of
 * remap_boxes_kernel for the one-lens tiles, the same for the rest}.  No reference counterpart.
 */
int pb_debug_plan_stage(const pb_plan *plan, int32_t out[8]);

#ifdef __cplusplus
}
#endif
#endif /* PB_REMAP_H */
