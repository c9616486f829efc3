// pb_device.cuh -- per-pixel float64 device math of the remap path (sm_100a).
//
// One output pixel goes through: output ray (a1/a3/a4 of SURVEY.md section 8) -> 0..n rotations
// (a7) -> source lookup (a9/a10/a11).  Everything here is float64 without FMA contraction
// (compiled with -fmad=false; the explicit __dmul_rn/__dadd_rn calls document where the
// reference rounds a product before it adds), because the truncated source index has to match
// the reference's NumPy float64 arithmetic bit for bit.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "pb_remap.h"

namespace pb {

constexpr double kPi = 3.141592653589793;  // == numpy.pi

// ---------------------------------------------------------------------------------- parameters

// Output geometry with the constants the reference derives from it, computed once on the host
// in the reference's own order of operations (see derive_out in pb_remap.cu).
struct OutGeom {
    int kind, lens;
    int H, W;      // W = effective output width (2*(width/2) for a double image)
    int half_w;    // double: width of one half
    double f;      // pixels per focal unit
    double half_fov;      // fov / 2: rays beyond it are invalid            projection.py:160, 357
    double right_lat_min; // double, right half: pi - fov/2                 projection.py:358-360
    // pixel-grid axes as numpy.linspace(start, stop, n): value(i) = fl(fl(i*step) + start), last == stop
    double x_start, x_stop, x_step;  // camera/double: x of a column        projection.py:177, 390-392
    double y_start, y_stop, y_step;  // camera/double: y of a row           projection.py:178-180, 399-401
                                     // equirect: x = longitude, y = latitude projection.py:502-505
    const double* lut;               // PB_LENS_TABLE: device samples of the reverse lens function
    double lut_scale;                // (n - 1) / x_max
    int lut_n;
};

struct SrcGeom {
    int kind, lens;
    int H, W, C;
    int wl, wr;           // double: widths of the left / right halves      projection.py:413, 429-431
    double f;
    double cy, cx;        // camera image centre (H/2-.5, W/2-.5)            projection.py:262-274
    double cxl, cxr;      // double: centres of the two halves
    double rect_limit;    // to_radians(89), rectilinear forward domain      lens.py:97-98
    double seg_h, seg_w, half_w;  // equirect: pi/H, pi/(W/2), W/2           projection.py:538-543
    double mrg_lo, mrg_hi, mrg_hi_safe, mrg_span;  // double blend band      projection.py:414-418
    const double* lut;    // PB_LENS_TABLE: device samples of the forward lens function
    double lut_scale;     // (n - 1) / x_max
    int lut_n;
};

struct Rotations {
    int n;
    double m[PB_MAX_ROTATIONS][9];
};

// ---------------------------------------------------------------------------------- helpers

__device__ __forceinline__ double linspace_at(double start, double stop, double step, int n, int i) {
    if (i == n - 1 && n > 1) return stop;
    return __dadd_rn(__dmul_rn((double)i, step), start);
}

// _shared.py:25-55 + np.log(z).imag: both parts are broadcast as x + y*0, y + x*0 first (this
// turns a lone -0.0 into +0.0 and spreads NaN), then the angle is atan2.
__device__ __forceinline__ double angle_of(double x, double y) {
    double fx = __dadd_rn(x, __dmul_rn(y, 0.0));
    double fy = __dadd_rn(y, __dmul_rn(x, 0.0));
    return atan2(fy, fx);
}

// ndarray.astype(int) on x86 (cvttsd2si): truncation toward zero; NaN and out-of-range give
// INT64_MIN.
__device__ __forceinline__ long long trunc_i64(double v) {
    if (!(fabs(v) < 9223372036854775808.0)) return (long long)0x8000000000000000ULL;
    return __double2ll_rz(v);
}

// numpy's % on int64 (sign of the divisor)
__device__ __forceinline__ long long floor_mod(long long a, long long m) {
    long long r = a % m;
    if (r != 0 && ((r < 0) != (m < 0))) r += m;
    return r;
}

// ---------------------------------------------------------------------------------- lenses

// A user-defined lens function from its table of samples (PB_LENS_TABLE): linear interpolation,
// x clamped to the table's range; NaN stays NaN.
__device__ __forceinline__ double lens_table_at(const double* __restrict__ lut, double scale, int n, double x) {
    if (x != x) return x;
    double t = x * scale;
    t = t < 0.0 ? 0.0 : t;
    int i = t >= (double)(n - 1) ? n - 2 : (int)t;
    const double a = __ldg(lut + i), b = __ldg(lut + i + 1);
    const double fr = fmin(t - (double)i, 1.0);
    return a + (b - a) * fr;
}

// lens.py:75-103, 126-144, 168-187, 224-243, 266-286, 313-335 (array branch)
__device__ __forceinline__ double lens_forward(const SrcGeom& s, double theta) {
    const int lens = s.lens;
    const double rect_limit = s.rect_limit;
    if (lens == PB_LENS_TABLE) return lens_table_at(s.lut, s.lut_scale, s.lut_n, theta);
    switch (lens) {
        case PB_LENS_EQUIDISTANT: return theta;
        case PB_LENS_EQUISOLID: return 2.0 * sin(theta / 2.0);
        case PB_LENS_ORTHOGRAPHIC: return sin(theta);
        case PB_LENS_STEREOGRAPHIC: return 2.0 * tan(theta / 2.0);
        case PB_LENS_RECTILINEAR:
            if (theta < 0.0 || theta > rect_limit) return __longlong_as_double(0x7ff8000000000000LL);
            return tan(theta);
        default: return __dmul_rn(1.47, sin(__dmul_rn(0.713, theta)));
    }
}

// lens.py:68-72, 106-124, 147-165, 190-220, 246-262, 289-309
__device__ __forceinline__ double lens_inverse(const OutGeom& g, double d) {
    const int lens = g.lens;
    if (lens == PB_LENS_TABLE) return lens_table_at(g.lut, g.lut_scale, g.lut_n, d);
    switch (lens) {
        case PB_LENS_EQUIDISTANT: return d;
        case PB_LENS_EQUISOLID: {
            double t = 2.0 * asin(d / 2.0);
            return (t != t) ? 0.0 : t;  // out-of-domain radius -> latitude 0 (and valid)
        }
        case PB_LENS_ORTHOGRAPHIC: return asin(d);
        case PB_LENS_STEREOGRAPHIC: return 2.0 * atan(d / 2.0);
        case PB_LENS_RECTILINEAR: return atan(d);
        default: return __ddiv_rn(asin(__ddiv_rn(d, 1.47)), 0.713);
    }
}

// ---------------------------------------------------------------------------------- rays

struct Ray {
    double lat, lon;
    bool invalid;
};

// a1 projection.py:487-513, a3 projection.py:147-194, a4 projection.py:341-406
template <int OUT_KIND>
__device__ __forceinline__ Ray output_ray(const OutGeom& g, int i, int j) {
    Ray r;
    if (OUT_KIND == PB_KIND_EQUIRECT) {
        r.lon = linspace_at(g.x_start, g.x_stop, g.x_step, g.W, j);
        r.lat = linspace_at(g.y_start, g.y_stop, g.y_step, g.H, i);
        r.invalid = false;
    } else {
        const bool right = (OUT_KIND == PB_KIND_DOUBLE) && j >= g.half_w;
        const int n_cols = (OUT_KIND == PB_KIND_DOUBLE) ? g.half_w : g.W;
        double x = linspace_at(g.x_start, g.x_stop, g.x_step, n_cols, right ? j - g.half_w : j);
        if (right) x = __dmul_rn(x, -1.0);
        const double y = linspace_at(g.y_start, g.y_stop, g.y_step, g.H, i);
        const double d = __ddiv_rn(sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y))), g.f);
        double lat = lens_inverse(g, d);
        if (right) {
            lat = __dadd_rn(__dmul_rn(lat, -1.0), kPi);
            r.invalid = lat < g.right_lat_min;
        } else {
            r.invalid = lat > g.half_fov;
        }
        r.lat = lat;
        r.lon = angle_of(x, y);
    }
    return r;
}

// a7 rotation.py:102-176 for one ray; m is row-major 3x3.
__device__ __forceinline__ Ray rotate_ray(Ray in, const double* __restrict__ m) {
    Ray out;
    out.invalid = in.invalid;
    if (in.invalid) {
        out.lat = 0.0;
        out.lon = 0.0;
        return out;
    }
    double sl, cl, so, co;
    sincos(in.lat, &sl, &cl);
    sincos(in.lon, &so, &co);
    const double vx = __dmul_rn(co, sl);
    const double vy = cl;
    const double vz = __dmul_rn(so, sl);
    const double nx = __dadd_rn(__dadd_rn(__dmul_rn(m[0], vx), __dmul_rn(m[1], vy)), __dmul_rn(m[2], vz));
    const double ny = __dadd_rn(__dadd_rn(__dmul_rn(m[3], vx), __dmul_rn(m[4], vy)), __dmul_rn(m[5], vz));
    const double nz = __dadd_rn(__dadd_rn(__dmul_rn(m[6], vx), __dmul_rn(m[7], vy)), __dmul_rn(m[8], vz));
    out.lat = acos(ny);
    out.lon = angle_of(nx, nz);
    return out;
}

// ---------------------------------------------------------------------------------- source lookup

// What one output pixel reads: up to two source pixels, each as packed coordinates
// (row << 16 | column, column already including the half offset / mirror of a double image;
// -1 = none, i.e. black) and their float64 weights.  Camera / equirect sources only use slot 0.
struct Lookup {
    int xy0, xy1;
    double w0, w1;
};

constexpr int kNoPixel = -1;

// ndarray.astype(int) followed by the bounds test of projection.py:223-231, for one coordinate:
// truncation toward zero BEFORE the test, so a coordinate in (-1, 0) lands on index 0 and is
// valid; NaN / inf / anything outside [0, n) is a "problem position" (-1).
// |v| + 2^52 rounded toward zero leaves trunc(|v|) in the low mantissa word (one DADD instead
// of a slow F2I.F64 conversion).
__device__ __forceinline__ int trunc_index(double v, int n) {
    const int hi = __double2hiint(v);
    const unsigned ahi = (unsigned)hi & 0x7fffffffu;
    const int idx = __double2loint(__dadd_rz(fabs(v), 4503599627370496.0));
    const bool ok = ahi < 0x41E00000u /* |v| < 2^31, not NaN */ && (unsigned)idx < (unsigned)n &&
                    !(hi < 0 && idx != 0);
    return ok ? idx : -1;
}

__device__ __forceinline__ int pack_xy(int px, int py, int col0, int w, bool flip) {
    if ((px | py) < 0) return kNoPixel;
    return (py << 16) | (col0 + (flip ? (w - 1 - px) : px));
}

// a9 projection.py:247-274 + 223-231 with the radius already known: cos/sin of the longitude
// and dist = forward_lens(lat) * f_distance.
__device__ __forceinline__ int camera_xy_from(double c, double s, double dist, int h, int w, double cy,
                                              double cx, int col0, bool flip) {
    const double fx = __dadd_rn(__dmul_rn(c, dist), cx);
    const double fy = __dadd_rn(__dmul_rn(__dmul_rn(s, dist), -1.0), cy);
    return pack_xy(trunc_index(fx, w), trunc_index(fy, h), col0, w, flip);
}

__device__ __forceinline__ int camera_xy(const SrcGeom& g, int h, int w, double cy,
                                         double cx, double lat, double lon, int col0, bool flip) {
    const double dist = __dmul_rn(lens_forward(g, lat), g.f);
    double s, c;
    sincos(lon, &s, &c);
    return camera_xy_from(c, s, dist, h, w, cy, cx, col0, flip);
}

// a10 projection.py:439-456
__device__ __forceinline__ double merge_weight(const SrcGeom& s, double lat) {
    if (lat >= s.mrg_lo && lat <= s.mrg_hi_safe) return __dmul_rn(__ddiv_rn(__dadd_rn(lat, -s.mrg_hi), s.mrg_span), -1.0);
    return 1.0;
}

// a11 projection.py:542-545 for one axis: trunc(v) mod n with Python's sign convention
__device__ __forceinline__ int wrap_index(double v, int n) {
    if (v >= 0.0 && v < 2147483648.0) {
        int t = __double2loint(__dadd_rz(v, 4503599627370496.0));
        if (t >= n) t = (t < 2 * n) ? t - n : t % n;
        return t;
    }
    return (int)floor_mod(trunc_i64(v), (long long)n);
}

template <int SRC_KIND>
__device__ __forceinline__ Lookup source_lookup(const SrcGeom& s, Ray r) {
    Lookup L;
    L.xy0 = L.xy1 = kNoPixel;
    L.w0 = L.w1 = 1.0;
    if (r.invalid) return L;
    if (SRC_KIND == PB_KIND_CAMERA) {
        L.xy0 = camera_xy(s, s.H, s.W, s.cy, s.cx, r.lat, r.lon, 0, false);
    } else if (SRC_KIND == PB_KIND_EQUIRECT) {
        // a11 projection.py:515-547: true division, truncation, Python-sign modulo
        const int row = wrap_index(__ddiv_rn(r.lat, s.seg_h), s.H);
        const int col = wrap_index(__dadd_rn(__ddiv_rn(r.lon, s.seg_w), s.half_w), s.W);
        L.xy0 = (row << 16) | col;
    } else {
        // a10 projection.py:408-462: both halves are sampled as plain cameras of magnitude H/2
        const double lat_l = r.lat;
        const double lat_r = __dadd_rn(__dmul_rn(r.lat, -1.0), kPi);
        double sn, cs;
        sincos(r.lon, &sn, &cs);
        const double dist_l = __dmul_rn(lens_forward(s, lat_l), s.f);
        const double dist_r = __dmul_rn(lens_forward(s, lat_r), s.f);
        L.xy0 = camera_xy_from(cs, sn, dist_l, s.H, s.wl, s.cy, s.cxl, 0, false);
        L.xy1 = camera_xy_from(cs, sn, dist_r, s.H, s.wr, s.cy, s.cxr, s.wl, true);
        L.w0 = merge_weight(s, lat_l);
        L.w1 = merge_weight(s, lat_r);
    }
    return L;
}

__device__ __forceinline__ int xy_to_offset(int xy, int width) {
    return xy < 0 ? -1 : (xy >> 16) * width + (xy & 0xffff);
}

// numpy's float64 -> uint8 cast on x86-64: truncation to a 32-bit integer (cvttsd2si), low byte
// kept; NaN and |v| >= 2^31 give 0x80000000, whose low byte is 0
__device__ __forceinline__ unsigned char cast_u8(double v) {
    if (!(fabs(v) < 2147483648.0)) return 0;
    return (unsigned char)(__double2int_rz(v) & 0xff);
}

// (left*wl + right*wr).astype(np.uint8)  (projection.py:459)
__device__ __forceinline__ unsigned char blend_u8(unsigned a, double wa, unsigned b, double wb) {
    return cast_u8(__dadd_rn(__dmul_rn((double)a, wa), __dmul_rn((double)b, wb)));
}

// ---------------------------------------------------------------------------------- typed blend
//
// A double-fisheye source that keeps its dtype (pb_plan_remap_typed ...): the reference's blend
// with its final cast to uint8 replaced by a cast to the source's own element type,
//     (left.astype(float64) * wl + right.astype(float64) * wr).astype(image.dtype)
// Elements travel as raw bits, zero-extended to 64; the type code (PB_ELEM_*) is uniform over a
// launch, so its switches do not diverge.

__host__ __device__ __forceinline__ int elem_type_bytes(int type) {
    switch (type) {
        case PB_ELEM_UINT8: case PB_ELEM_INT8: case PB_ELEM_BOOL: return 1;
        case PB_ELEM_UINT16: case PB_ELEM_INT16: case PB_ELEM_FLOAT16: case PB_ELEM_BFLOAT16: return 2;
        case PB_ELEM_UINT32: case PB_ELEM_INT32: case PB_ELEM_FLOAT32: return 4;
        case PB_ELEM_UINT64: case PB_ELEM_INT64: case PB_ELEM_FLOAT64: return 8;
        default: return 0;
    }
}

// ndarray.astype(float64) of one element: exact for every type but the 64-bit integers, which
// round to nearest (cvtsi2sd, and gcc's uint64 sequence, on x86-64)
__device__ __forceinline__ double elem_to_f64(unsigned long long bits, int type) {
    switch (type) {
        case PB_ELEM_INT8: return (double)(signed char)bits;
        case PB_ELEM_BOOL: return (bits & 0xffu) != 0 ? 1.0 : 0.0;
        case PB_ELEM_UINT16: return (double)(unsigned short)bits;
        case PB_ELEM_INT16: return (double)(short)bits;
        case PB_ELEM_FLOAT16: {
            double d;
            asm("cvt.f64.f16 %0, %1;" : "=d"(d) : "h"((unsigned short)bits));
            return d;
        }
        case PB_ELEM_BFLOAT16: return (double)__uint_as_float((unsigned)bits << 16);
        case PB_ELEM_UINT32: return (double)(unsigned)bits;
        case PB_ELEM_INT32: return (double)(int)(unsigned)bits;
        case PB_ELEM_FLOAT32: return (double)__uint_as_float((unsigned)bits);
        case PB_ELEM_UINT64: return __ull2double_rn(bits);
        case PB_ELEM_INT64: return __ll2double_rn((long long)bits);
        case PB_ELEM_FLOAT64: return __longlong_as_double((long long)bits);
        default: return (double)(unsigned char)bits;
    }
}

// ndarray.astype(type) of one float64 on x86-64 (NumPy's casts, bfloat16: torch's):
//   8 / 16-bit integers  truncation to int32 (cvttsd2si), low bits kept; NaN, |v| >= 2^31 -> 0
//   int32 / int64        truncation; NaN and out of range -> INT32_MIN / INT64_MIN
//   uint32               truncation to int64, low 32 bits kept
//   uint64               v < 2^63 (or NaN): truncation to int64; else trunc(v - 2^63) ^ 2^63
//   float32 / float16    ONE rounding to nearest even (float16 straight from float64)
//   bfloat16             two: to float32, then to bfloat16, both to nearest even
//   bool                 v != 0 (NaN is True)
__device__ __forceinline__ unsigned long long f64_to_elem(double v, int type) {
    switch (type) {
        case PB_ELEM_BOOL: return v != 0.0 ? 1ull : 0ull;
        case PB_ELEM_UINT16: case PB_ELEM_INT16:
            return fabs(v) < 2147483648.0 ? (unsigned long long)(__double2int_rz(v) & 0xffff) : 0ull;
        case PB_ELEM_FLOAT16: {
            unsigned short h;
            asm("cvt.rn.f16.f64 %0, %1;" : "=h"(h) : "d"(v));
            return h;
        }
        case PB_ELEM_BFLOAT16: {
            unsigned short h;
            asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(h) : "f"(__double2float_rn(v)));
            return h;
        }
        case PB_ELEM_INT32:
            return (unsigned)(v > -2147483649.0 && v < 2147483648.0 ? __double2int_rz(v) : (int)0x80000000u);
        case PB_ELEM_UINT32: return (unsigned)(unsigned long long)trunc_i64(v);
        case PB_ELEM_FLOAT32: return __float_as_uint(__double2float_rn(v));
        case PB_ELEM_INT64: return (unsigned long long)trunc_i64(v);
        case PB_ELEM_UINT64:
            if (!(v >= 9223372036854775808.0)) return (unsigned long long)trunc_i64(v);
            return (unsigned long long)trunc_i64(__dadd_rn(v, -9223372036854775808.0)) ^ 0x8000000000000000ull;
        case PB_ELEM_FLOAT64: return (unsigned long long)__double_as_longlong(v);
        default: return cast_u8(v);  // uint8, int8
    }
}

// One element of the blend: the products are rounded before the sum (no FMA, as blend_u8); a lens
// without a sample contributes 0 * its weight
__device__ __forceinline__ unsigned long long blend_elem(unsigned long long a, double wa, unsigned long long b, double wb,
                                                         int type) {
    return f64_to_elem(__dadd_rn(__dmul_rn(elem_to_f64(a, type), wa), __dmul_rn(elem_to_f64(b, type), wb)), type);
}

// raw element of `bytes` (1, 2, 4, 8) bytes at p, zero-extended; and the store of its low bytes
__device__ __forceinline__ unsigned long long load_elem(const unsigned char* p, int bytes) {
    switch (bytes) {
        case 1: return __ldg(p);
        case 2: return __ldg(reinterpret_cast<const unsigned short*>(p));
        case 4: return __ldg(reinterpret_cast<const unsigned*>(p));
        default: return __ldg(reinterpret_cast<const unsigned long long*>(p));
    }
}
__device__ __forceinline__ void store_elem(unsigned char* p, int bytes, unsigned long long v) {
    switch (bytes) {
        case 1: *p = (unsigned char)v; break;
        case 2: *reinterpret_cast<unsigned short*>(p) = (unsigned short)v; break;
        case 4: *reinterpret_cast<unsigned*>(p) = (unsigned)v; break;
        default: *reinterpret_cast<unsigned long long*>(p) = v; break;
    }
}

// One pixel of C elements of a double-fisheye source, element type `type`: p0 / p1 the two lenses'
// pixels (null: no sample), o the output pixel
__device__ __forceinline__ void blend_px_typed(const unsigned char* p0, double w0, const unsigned char* p1, double w1,
                                               unsigned char* o, int C, int type) {
    const int E = elem_type_bytes(type);
    for (int c = 0; c < C; ++c) {
        const unsigned long long v0 = p0 ? load_elem(p0 + c * E, E) : 0ull;
        const unsigned long long v1 = p1 ? load_elem(p1 + c * E, E) : 0ull;
        store_elem(o + c * E, E, blend_elem(v0, w0, v1, w1, type));
    }
}

}  // namespace pb
