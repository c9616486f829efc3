/*
 * pb_oracle.c -- scalar float64 C restatement of photonbend's per-pixel remap path.
 *
 * TEST INFRASTRUCTURE ONLY.  This is the checker, never the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline leg may load it.  The product
 * (photonbend_b200) never links, imports or executes anything under oracle/.
 *
 * It follows the reference (/root/reference/photonbend, pure Python + NumPy) one
 * output pixel at a time, keeping every polar round trip the reference makes
 * (angles -> unit vector -> rotate -> angles, once per rotation) and the reference's
 * evaluation order, with glibc libm for the transcendentals.  NumPy itself evaluates
 * cos/sin of a longitude through cexp() and atan2 through clog(), i.e. through the
 * same glibc routines used here; np.cos/np.sin/np.arccos/np.arcsin/np.arctan/np.tan on
 * real arrays go through NumPy's own SIMD kernels, which differ from glibc in the last
 * ulp.  Those ulp differences do not reach the truncated pixel index in any golden
 * vector (tests/test_oracle_golden.py pins this file against tests/golden/, generated
 * from the live reference by tests/golden/make_golden.py); oracle/numpy_port.py is the
 * bit-identical-by-construction twin.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -shared).  Single-threaded C: the
 * ctypes front-end (oracle/c_port.py) runs row bands on a thread pool (ctypes drops the GIL).
 * -ffp-contract=off matters: the reference never fuses a multiply with an add.
 */
#include <math.h>
#include <stdint.h>
#include <stddef.h>
#include <string.h>

enum { PBO_CAMERA = 0, PBO_DOUBLE = 1, PBO_EQUIRECT = 2 };
enum {
    PBO_EQUIDISTANT = 0,
    PBO_EQUISOLID = 1,
    PBO_ORTHOGRAPHIC = 2,
    PBO_STEREOGRAPHIC = 3,
    PBO_RECTILINEAR = 4,
    PBO_THOBY = 5
};

typedef struct pbo_image {
    int32_t kind;      /* PBO_CAMERA / PBO_DOUBLE / PBO_EQUIRECT */
    int32_t lens;      /* PBO_* lens id (ignored for equirect) */
    int32_t height;
    int32_t width;
    double fov;        /* camera: full field of view; double: per-sensor fov (radians) */
    double f_distance; /* pixels per focal unit, derived by the caller exactly as the
                          reference does (projection.py:141-144, 336-339) */
} pbo_image;

static const double PI = 3.141592653589793; /* == numpy.pi */

/* utils/__init__.py:27-37 */
static double to_radians(double deg) { return deg / 180 * PI; }

/* lens.py:75-103, 126-144, 168-187, 224-243, 266-286, 313-335 (array branch) */
static double lens_forward(int lens, double theta)
{
    switch (lens) {
    case PBO_EQUIDISTANT:
        return theta;
    case PBO_EQUISOLID:
        return 2 * sin(theta / 2.0);
    case PBO_ORTHOGRAPHIC:
        return sin(theta);
    case PBO_STEREOGRAPHIC:
        return 2.0 * tan(theta / 2.0);
    case PBO_RECTILINEAR:
        if (theta < 0 || theta > to_radians(89))
            return NAN;
        return tan(theta);
    case PBO_THOBY:
        return 1.47 * sin(0.713 * theta);
    }
    return NAN;
}

/* lens.py:68-72, 106-124, 147-165, 190-220, 246-262, 289-309 */
static double lens_inverse(int lens, double d)
{
    double t;
    switch (lens) {
    case PBO_EQUIDISTANT:
        return d;
    case PBO_EQUISOLID:
        t = 2.0 * asin(d / 2.0);
        return isnan(t) ? 0.0 : t;
    case PBO_ORTHOGRAPHIC:
        return asin(d);
    case PBO_STEREOGRAPHIC:
        return 2.0 * atan(d / 2.0);
    case PBO_RECTILINEAR:
        return atan(d);
    case PBO_THOBY:
        return asin(d / 1.47) / 0.713;
    }
    return NAN;
}

/* numpy.linspace(start, stop, num)[i]: fl(fl(i*step)+start), last element == stop */
static double linspace_at(double start, double stop, int num, int i)
{
    if (num <= 1)
        return start;
    if (i == num - 1)
        return stop;
    double step = (stop - start) / (double)(num - 1);
    return (double)i * step + start;
}

/* x86 cvttsd2si semantics of ndarray.astype(int): NaN / out of range -> INT64_MIN */
static int64_t trunc_i64(double v)
{
    if (!(fabs(v) < 9223372036854775808.0))
        return INT64_MIN;
    return (int64_t)v;
}

/* Python-sign modulo, as numpy's % on int64 */
static int64_t floor_mod(int64_t a, int64_t m)
{
    int64_t r = a % m;
    if (r != 0 && ((r < 0) != (m < 0)))
        r += m;
    return r;
}

/* _shared.py:25-55 then np.log(...).imag: the two parts are first broadcast against each
 * other as x + y*0 and y + x*0 (which turns a -0.0 into +0.0 and spreads NaN/inf), and the
 * angle is the imaginary part of the complex log, i.e. atan2. */
static double angle_of(double x, double y)
{
    double fx = x + y * 0;
    double fy = y + x * 0;
    return atan2(fy, fx);
}

typedef struct ray {
    double lat, lon;
    int invalid;
} ray;

/* projection.py:487-513 */
static ray equirect_ray(const pbo_image *g, int i, int j)
{
    ray r;
    double half_px = PI / g->width / 2;
    r.lon = linspace_at(-PI + half_px, PI - half_px, g->width, j);
    r.lat = linspace_at(0, PI, g->height, i);
    r.invalid = 0;
    return r;
}

/* projection.py:147-194 */
static ray camera_ray(const pbo_image *g, int i, int j)
{
    ray r;
    double w = g->width, h = g->height;
    double x = linspace_at(-w / 2 + 0.5, w / 2 - 0.5, g->width, j);
    double y = linspace_at(h / 2 - 0.5, -h / 2 + 0.5, g->height, i);
    double d = sqrt(x * x + y * y) / g->f_distance;
    r.lat = lens_inverse(g->lens, d);
    r.lon = angle_of(x, y);
    r.invalid = r.lat > g->fov / 2;
    return r;
}

/* projection.py:341-406 */
static ray double_ray(const pbo_image *g, int i, int j)
{
    ray r;
    int hw = g->width / 2;
    double fhw = hw, h = g->height;
    int right = j >= hw;
    double x = linspace_at(-fhw / 2 + 0.5, fhw / 2 - 0.5, hw, right ? j - hw : j);
    if (right)
        x = x * (-1);
    double y = linspace_at(h / 2 - 0.5, -h / 2 + 0.5, g->height, i);
    double d = sqrt(x * x + y * y) / g->f_distance;
    r.lat = lens_inverse(g->lens, d);
    if (right) {
        r.lat = r.lat * -1;
        r.lat = r.lat + PI;
        r.invalid = r.lat < PI - (g->fov / 2.0);
    } else {
        r.invalid = r.lat > g->fov / 2.0;
    }
    r.lon = angle_of(x, y);
    return r;
}

static ray output_ray(const pbo_image *g, int i, int j)
{
    switch (g->kind) {
    case PBO_EQUIRECT:
        return equirect_ray(g, i, j);
    case PBO_CAMERA:
        return camera_ray(g, i, j);
    default:
        return double_ray(g, i, j);
    }
}

/* rotation.py:102-176 for one pixel; m is row-major 3x3 */
static ray rotate_ray(ray in, const double *m)
{
    ray out;
    if (in.invalid) {
        out.lat = 0;
        out.lon = 0;
        out.invalid = 1;
        return out;
    }
    double sl = sin(in.lat);
    double vy = cos(in.lat);
    double vx = cos(in.lon) * sl;
    double vz = sin(in.lon) * sl;
    double nx = (m[0] * vx + m[1] * vy) + m[2] * vz;
    double ny = (m[3] * vx + m[4] * vy) + m[5] * vz;
    double nz = (m[6] * vx + m[7] * vy) + m[8] * vz;
    out.lat = acos(ny);
    out.lon = angle_of(nx, nz);
    out.invalid = 0;
    return out;
}

/* projection.py:197-274: one camera sample.  Returns 1 and the pixel offset when the ray
 * lands inside the image, 0 ("problem position" -> black) otherwise. */
static int camera_lookup(int lens, double f, int h, int w, double lat, double lon,
                         int64_t *px, int64_t *py)
{
    double cy = (double)h / 2 - 0.5;
    double cx = (double)w / 2 - 0.5;
    double dist = lens_forward(lens, lat) * f;
    double re = cos(lon) * dist;
    double im = sin(lon) * dist;
    int64_t y = trunc_i64((im * (-1)) + cy);
    int64_t x = trunc_i64(re + cx);
    if (y >= h || y < 0 || x >= w || x < 0)
        return 0;
    *px = x;
    *py = y;
    return 1;
}

/* ndarray.astype(np.uint8) from float64 on x86-64: truncation to a 32-bit integer
 * (cvttsd2si), low byte kept; NaN and |v| >= 2^31 give INT32_MIN, whose low byte is 0 */
static uint8_t wrap_u8(double v)
{
    if (!(fabs(v) < 2147483648.0))
        return 0;
    return (uint8_t)((int32_t)v & 0xFF);
}

/* projection.py:439-456 */
static double merge_weight(double lat, double lo, double hi, double span, double safety)
{
    if (lat >= lo && lat <= (hi + safety))
        return (lat - hi) / span * -1;
    return 1.0;
}

static void sample_pixel(const pbo_image *s, const uint8_t *img, int channels, ray r,
                         uint8_t *dst)
{
    int c;
    if (s->kind == PBO_CAMERA) {
        /* projection.py:197-245 */
        int64_t px, py;
        if (!r.invalid &&
            camera_lookup(s->lens, s->f_distance, s->height, s->width, r.lat, r.lon, &px, &py)) {
            const uint8_t *p = img + ((size_t)py * s->width + px) * channels;
            for (c = 0; c < channels; ++c)
                dst[c] = p[c];
        } else {
            for (c = 0; c < channels; ++c)
                dst[c] = 0;
        }
    } else if (s->kind == PBO_EQUIRECT) {
        /* projection.py:515-547 */
        if (r.invalid) {
            for (c = 0; c < channels; ++c)
                dst[c] = 0;
            return;
        }
        double seg_w = PI / ((double)s->width / 2);
        double seg_h = PI / (double)s->height;
        double frow = r.lat / seg_h;
        double fcol = r.lon / seg_w + ((double)s->width / 2);
        int64_t row = floor_mod(trunc_i64(frow), s->height);
        int64_t col = floor_mod(trunc_i64(fcol), s->width);
        const uint8_t *p = img + ((size_t)row * s->width + col) * channels;
        for (c = 0; c < channels; ++c)
            dst[c] = p[c];
    } else {
        /* projection.py:408-462 */
        if (r.invalid) {
            for (c = 0; c < channels; ++c)
                dst[c] = 0;
            return;
        }
        int wl = s->width / 2;
        int wr = s->width - wl;
        double ref = (s->fov / 2) - (PI / 2);
        double lo = PI / 2 - ref;
        double hi = PI / 2 + ref;
        double span = 2.0 * ref;
        double safety = to_radians(0.5);
        double lat_l = r.lat;
        double lat_r = r.lat * -1;
        lat_r = lat_r + PI;
        int64_t px, py;
        const uint8_t *pl = NULL, *pr = NULL;
        if (camera_lookup(s->lens, s->f_distance, s->height, wl, lat_l, r.lon, &px, &py))
            pl = img + ((size_t)py * s->width + px) * channels;
        if (camera_lookup(s->lens, s->f_distance, s->height, wr, lat_r, r.lon, &px, &py))
            pr = img + ((size_t)py * s->width + (wl + (wr - 1 - px))) * channels; /* flipped half */
        double wgt_l = merge_weight(lat_l, lo, hi, span, safety);
        double wgt_r = merge_weight(lat_r, lo, hi, span, safety);
        for (c = 0; c < channels; ++c) {
            double a = (double)(pl ? pl[c] : 0) * wgt_l;
            double b = (double)(pr ? pr[c] : 0) * wgt_r;
            dst[c] = wrap_u8(a + b);
        }
    }
}

/* effective output width: a double output only has 2*(W//2) columns (projection.py:389-397) */
static int out_width(const pbo_image *g)
{
    return g->kind == PBO_DOUBLE ? 2 * (g->width / 2) : g->width;
}

/*
 * The reference's three-call protocol for output rows [row0, row1):
 *   dst.get_coordinate_map() -> Rotation.rotate_coordinate_map() x n_rot -> src.process_coordinate_map()
 * rot: n_rot row-major 3x3 matrices (Rotation.rotation_matrix), applied in order.
 * dst / map / idx are indexed by absolute row: row i is written at offset i*out_width*(...),
 * so disjoint bands of one full-size buffer can be filled from several threads.
 */
int pbo_remap_u8(const pbo_image *out, int n_rot, const double *rot, const pbo_image *src,
                 const uint8_t *src_pixels, int channels, uint8_t *dst, int row0, int row1)
{
    int wo = out_width(out);
    if (channels < 1 || row0 < 0 || row1 > out->height || row0 > row1)
        return 1;
    for (int i = row0; i < row1; ++i) {
        for (int j = 0; j < wo; ++j) {
            ray r = output_ray(out, i, j);
            for (int k = 0; k < n_rot; ++k)
                r = rotate_ray(r, rot + 9 * k);
            sample_pixel(src, src_pixels, channels, r,
                         dst + ((size_t)i * wo + j) * channels);
        }
    }
    return 0;
}

/* The coordinate map itself, float64 (H, W, 3) = (lat, lon, invalid), after n_rot rotations. */
int pbo_coordinate_map_f64(const pbo_image *out, int n_rot, const double *rot, double *map,
                           int row0, int row1)
{
    int wo = out_width(out);
    for (int i = row0; i < row1; ++i) {
        for (int j = 0; j < wo; ++j) {
            ray r = output_ray(out, i, j);
            for (int k = 0; k < n_rot; ++k)
                r = rotate_ray(r, rot + 9 * k);
            double *m = map + ((size_t)i * wo + j) * 3;
            m[0] = r.lat;
            m[1] = r.lon;
            m[2] = r.invalid ? 1.0 : 0.0;
        }
    }
    return 0;
}

/*
 * The source index map the remap resolves to, for roofline accounting and mismatch
 * attribution: idx[(i*W+j)*2 + {0,1}] = linear source pixel offsets of the (left, right)
 * samples, -1 where there is none (black).  Camera / equirect sources only fill slot 0.
 */
int pbo_source_index_i64(const pbo_image *out, int n_rot, const double *rot,
                         const pbo_image *src, int64_t *idx, int row0, int row1)
{
    int wo = out_width(out);
    for (int i = row0; i < row1; ++i) {
        for (int j = 0; j < wo; ++j) {
            ray r = output_ray(out, i, j);
            for (int k = 0; k < n_rot; ++k)
                r = rotate_ray(r, rot + 9 * k);
            int64_t *o = idx + ((size_t)i * wo + j) * 2;
            int64_t px, py;
            o[0] = o[1] = -1;
            if (r.invalid)
                continue;
            if (src->kind == PBO_CAMERA) {
                if (camera_lookup(src->lens, src->f_distance, src->height, src->width, r.lat,
                                  r.lon, &px, &py))
                    o[0] = py * src->width + px;
            } else if (src->kind == PBO_EQUIRECT) {
                double seg_w = PI / ((double)src->width / 2);
                double seg_h = PI / (double)src->height;
                int64_t row = floor_mod(trunc_i64(r.lat / seg_h), src->height);
                int64_t col = floor_mod(trunc_i64(r.lon / seg_w + ((double)src->width / 2)),
                                        src->width);
                o[0] = row * src->width + col;
            } else {
                int wl = src->width / 2, wr = src->width - wl;
                double lat_r = r.lat * -1;
                lat_r = lat_r + PI;
                if (camera_lookup(src->lens, src->f_distance, src->height, wl, r.lat, r.lon,
                                  &px, &py))
                    o[0] = py * src->width + px;
                if (camera_lookup(src->lens, src->f_distance, src->height, wr, lat_r, r.lon,
                                  &px, &py))
                    o[1] = py * src->width + (wl + (wr - 1 - px));
            }
        }
    }
    return 0;
}

int pbo_version(void) { return 1; }
