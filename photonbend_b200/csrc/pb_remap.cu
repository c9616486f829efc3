// pb_remap.cu -- kernels and C ABI of libpbremap.so (see include/pb_remap.h).
//
// Build (photonbend_b200/build.py):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false
//        -Xcompiler -fPIC,-ffp-contract=off -shared -Iinclude -o libpbremap.so pb_remap.cu
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "pb_device.cuh"
#include "pb_tiled.cuh"
#include "pb_sep1.cuh"
#include "pb_chunk.cuh"
#include "pb_tiled2.cuh"
#include "pb_wide.cuh"

namespace pb {

// ------------------------------------------------------------------------------------ errors

static thread_local std::string g_last_error;
// kernels this library has launched in this process (pb_kernel_launches)
static std::atomic<long long> g_kernel_launches{0};
#define PB_COUNT_LAUNCH() g_kernel_launches.fetch_add(1, std::memory_order_relaxed)

static int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

static int cuda_fail(cudaError_t e, const char* what) {
    return fail(PB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// ------------------------------------------------------------------------------------ host-side derivation
// Everything below is evaluated in the reference's order of operations; this translation unit's
// host code is compiled with -ffp-contract=off so no product is fused into a sum.

static double to_radians(double deg) { return deg / 180 * kPi; }  // utils/__init__.py:27-37

static double linspace_step(double start, double stop, int n) {
    return n > 1 ? (stop - start) / (double)(n - 1) : 0.0;
}

static int check_image(const pb_image_desc& d, const char* which) {
    if (d.kind < PB_KIND_CAMERA || d.kind > PB_KIND_EQUIRECT)
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(which) + ": unknown image kind");
    if (d.height < 1 || d.width < 1)
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(which) + ": height and width must be positive");
    if ((long long)d.height * (long long)d.width >= (1LL << 31))
        return fail(PB_ERR_UNSUPPORTED, std::string(which) + ": more than 2^31 pixels");
    if (d.kind != PB_KIND_EQUIRECT && (d.lens < PB_LENS_EQUIDISTANT || d.lens > PB_LENS_TABLE))
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(which) + ": unknown lens");
    if (d.kind != PB_KIND_EQUIRECT && d.lens == PB_LENS_TABLE &&
        (!d.lens_table || d.lens_table_n < 2 || d.lens_table_n > (1 << 24) || !(d.lens_table_max > 0.0) ||
         !std::isfinite(d.lens_table_max)))
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(which) + ": PB_LENS_TABLE needs lens_table (>= 2 samples) and lens_table_max > 0");
    if (d.kind == PB_KIND_DOUBLE && d.width < 2)
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(which) + ": a double image needs width >= 2");
    return PB_OK;
}

static OutGeom derive_out(const pb_image_desc& d) {
    OutGeom g;
    std::memset(&g, 0, sizeof(g));
    g.kind = d.kind;
    g.lens = d.lens;
    g.H = d.height;
    g.W = d.width;
    g.f = d.f_distance;
    const double h = (double)d.height;
    if (d.kind == PB_KIND_EQUIRECT) {
        // projection.py:499-505
        const double w = (double)d.width;
        const double half_px = kPi / w / 2;
        g.x_start = -kPi + half_px;
        g.x_stop = kPi - half_px;
        g.x_step = linspace_step(g.x_start, g.x_stop, d.width);
        g.y_start = 0.0;
        g.y_stop = kPi;
        g.y_step = linspace_step(g.y_start, g.y_stop, d.height);
    } else {
        int cols = d.width;
        if (d.kind == PB_KIND_DOUBLE) {
            // projection.py:355-360, 389-401
            g.half_w = d.width / 2;
            g.W = 2 * g.half_w;
            cols = g.half_w;
            g.right_lat_min = kPi - (d.fov / 2.0);
        }
        const double w = (double)cols;
        g.half_fov = d.fov / 2;
        g.x_start = -w / 2 + 0.5;  // projection.py:177
        g.x_stop = w / 2 - 0.5;
        g.x_step = linspace_step(g.x_start, g.x_stop, cols);
        g.y_start = h / 2 - 0.5;   // projection.py:178-180
        g.y_stop = -h / 2 + 0.5;
        g.y_step = linspace_step(g.y_start, g.y_stop, d.height);
    }
    return g;
}

static SrcGeom derive_src(const pb_image_desc& d, int channels) {
    SrcGeom s;
    std::memset(&s, 0, sizeof(s));
    s.kind = d.kind;
    s.lens = d.lens;
    s.H = d.height;
    s.W = d.width;
    s.C = channels;
    s.f = d.f_distance;
    s.rect_limit = to_radians(89);
    const double h = (double)d.height, w = (double)d.width;
    s.cy = h / 2 - 0.5;  // projection.py:274
    s.cx = w / 2 - 0.5;
    if (d.kind == PB_KIND_EQUIRECT) {
        s.seg_w = kPi / (w / 2);  // projection.py:539-543
        s.seg_h = kPi / h;
        s.half_w = w / 2;
    } else if (d.kind == PB_KIND_DOUBLE) {
        s.wl = d.width / 2;       // projection.py:413
        s.wr = d.width - s.wl;
        s.cxl = (double)s.wl / 2 - 0.5;
        s.cxr = (double)s.wr / 2 - 0.5;
        const double ref = (d.fov / 2) - (kPi / 2);  // projection.py:414-418
        s.mrg_lo = kPi / 2 - ref;
        s.mrg_hi = kPi / 2 + ref;
        s.mrg_span = 2.0 * ref;
        s.mrg_hi_safe = s.mrg_hi + to_radians(0.5);
    }
    return s;
}

static bool has_table(const pb_image_desc& d) { return d.kind != PB_KIND_EQUIRECT && d.lens == PB_LENS_TABLE; }

// Device copies of the lens tables of a remap (PB_LENS_TABLE), one allocation: *dev owns them.
// The host tables are pageable memory: the copies are staged before the call returns, so the caller
// may free its tables afterwards.
static cudaError_t upload_lens_tables(const pb_image_desc* od, OutGeom* og, const pb_image_desc* sd, SrcGeom* sg,
                                      double** dev, cudaStream_t st, bool stream_ordered) {
    *dev = nullptr;
    const size_t n_out = (od && og && has_table(*od)) ? (size_t)od->lens_table_n : 0;
    const size_t n_src = (sd && sg && has_table(*sd)) ? (size_t)sd->lens_table_n : 0;
    if (n_out + n_src == 0) return cudaSuccess;
    cudaError_t e = stream_ordered ? cudaMallocAsync((void**)dev, (n_out + n_src) * sizeof(double), st)
                                   : cudaMalloc((void**)dev, (n_out + n_src) * sizeof(double));
    if (e != cudaSuccess) return e;
    if (n_out) {
        e = cudaMemcpyAsync(*dev, od->lens_table, n_out * sizeof(double), cudaMemcpyHostToDevice, st);
        og->lut = *dev;
        og->lut_n = (int)n_out;
        og->lut_scale = (double)(n_out - 1) / od->lens_table_max;
    }
    if (n_src && e == cudaSuccess) {
        e = cudaMemcpyAsync(*dev + n_out, sd->lens_table, n_src * sizeof(double), cudaMemcpyHostToDevice, st);
        sg->lut = *dev + n_out;
        sg->lut_n = (int)n_src;
        sg->lut_scale = (double)(n_src - 1) / sd->lens_table_max;
    }
    if (e != cudaSuccess) {
        if (stream_ordered) cudaFreeAsync(*dev, st);
        else cudaFree(*dev);
        *dev = nullptr;
    }
    return e;
}

// Constants of the guarded short cut (pb_fast.cuh).  Nothing here has to be bit-identical to
// the reference: these are decision thresholds with a guard band, not values that reach a pixel.
static FastGeom derive_fast(const pb_image_desc& od, const OutGeom& o, const pb_image_desc& sd, const SrcGeom& s,
                            int n_rot, const double (*rotations)[9]) {
    FastGeom g;
    std::memset(&g, 0, sizeof(g));
    const double inf = INFINITY;
    const double rel = 1e-9;  // relative guard on angles and radii
    g.n_rot = n_rot;
    g.enabled = 1;
    if (has_table(od) || has_table(sd)) g.enabled = 0;  // a user-defined lens has no algebraic form: exact chain
    // R_total = R_n ... R_1: the short cut applies all rotations as one matrix
    double acc[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int k = 0; k < n_rot; ++k) {
        double nxt[9];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)
                nxt[3 * r + c] = rotations[k][3 * r] * acc[c] + rotations[k][3 * r + 1] * acc[3 + c] +
                                 rotations[k][3 * r + 2] * acc[6 + c];
        std::memcpy(acc, nxt, sizeof(acc));
    }
    g.has_rot = n_rot > 0;
    std::memcpy(g.rot, acc, sizeof(acc));
    for (int e = 0; e < 9; ++e)
        if (!std::isfinite(acc[e])) g.enabled = 0;
    // The short cut carries the ray as a unit vector through ONE composed matrix; the exact chain
    // goes back to (acos, atan2) after every rotation.  The two are the same function only for
    // orthonormal matrices (Rotation.rotation_matrix always is; the raw ABI takes any 9 doubles):
    // anything else runs the exact chain.
    for (int k = 0; k < n_rot; ++k)
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) {
                double dot = 0.0;
                for (int e = 0; e < 3; ++e) dot += rotations[k][3 * r + e] * rotations[k][3 * c + e];
                if (!(std::fabs(dot - (r == c ? 1.0 : 0.0)) < 1e-12)) g.enabled = 0;
            }
    if (const char* e = std::getenv("PB_EXACT_CHAIN")) {  // validation: every pixel through the exact chain
        if (std::atoi(e) != 0) g.enabled = 0;
    }
    g.r2_valid = g.r2_invalid = g.r2_domain = inf;
    if (o.kind != PB_KIND_EQUIRECT) {
        const double f = o.f, hf = o.half_fov;
        if (!(f > 0.0) || !std::isfinite(f) || !std::isfinite(hf)) g.enabled = 0;
        g.inv_f = 1.0 / f;
        // radius (in focal units) at which the latitude crosses fov / 2; inf = never
        double d_star = inf;
        switch (o.lens) {
            case PB_LENS_EQUIDISTANT: d_star = hf; break;
            case PB_LENS_EQUISOLID: d_star = hf < kPi ? 2.0 * std::sin(hf / 2.0) : inf; break;
            case PB_LENS_ORTHOGRAPHIC: d_star = hf < kPi / 2 ? std::sin(hf) : inf; break;
            case PB_LENS_STEREOGRAPHIC: d_star = hf < kPi ? 2.0 * std::tan(hf / 2.0) : inf; break;
            case PB_LENS_RECTILINEAR: d_star = hf < kPi / 2 ? std::tan(hf) : inf; break;
            default: d_star = 0.713 * hf < kPi / 2 ? 1.47 * std::sin(0.713 * hf) : inf; break;
        }
        if (hf < 0.0) {  // every ray is outside the fov
            g.r2_valid = -1.0;
            g.r2_invalid = -1.0;
        } else if (d_star < inf) {
            const double r_star = d_star * f;
            g.r2_valid = (r_star * (1.0 - rel)) * (r_star * (1.0 - rel));
            g.r2_invalid = (r_star * (1.0 + rel)) * (r_star * (1.0 + rel));
        }
        // edge of the well-conditioned part of the lens inverse's domain
        const double edge = 1.0 - 1e-6;
        switch (o.lens) {
            case PB_LENS_EQUISOLID: g.r2_domain = 4.0 * f * f * edge; break;
            case PB_LENS_ORTHOGRAPHIC: g.r2_domain = f * f * edge; break;
            case PB_LENS_THOBY: g.r2_domain = 1.47 * 1.47 * f * f * edge; break;
            case PB_LENS_EQUIDISTANT:
                // without a rotation the latitude reaches the source as it is, not through acos
                if (n_rot == 0) g.r2_domain = (kPi * (1.0 - rel) * f) * (kPi * (1.0 - rel) * f);
                break;
            default: break;
        }
    }
    g.src_f = s.f;
    g.ny_rect_in = g.ny_rect_out = 0.0;
    g.ny_band_lo = 2.0;
    g.ny_band_hi = -2.0;
    if (s.kind == PB_KIND_EQUIRECT) {
        g.inv_seg_h = 1.0 / s.seg_h;
        g.inv_seg_w = 1.0 / s.seg_w;
    } else {
        if (!(s.f > 0.0) || !std::isfinite(s.f)) g.enabled = 0;
        const double c = std::cos(s.rect_limit);
        g.ny_rect_in = c * (1.0 + rel);
        g.ny_rect_out = c * (1.0 - rel);
        if (s.kind == PB_KIND_DOUBLE) {
            if (!std::isfinite(s.mrg_lo) || !std::isfinite(s.mrg_hi_safe)) g.enabled = 0;
            if (s.mrg_lo <= s.mrg_hi_safe) {
                // latitudes at which either lens may get a weight != 1 (projection.py:439-456):
                // lat in [lo, hi_safe] (left) or pi - lat in [lo, hi_safe] (right)
                const double t_lo = std::fmin(s.mrg_lo, kPi - s.mrg_hi_safe) - rel;
                const double t_hi = std::fmax(s.mrg_hi_safe, kPi - s.mrg_lo) + rel;
                g.ny_band_hi = std::cos(std::fmax(t_lo, 0.0)) + rel;
                g.ny_band_lo = std::cos(std::fmin(t_hi, kPi)) - rel;
            }
        }
    }
    return g;
}

// Constants of the FP32-first tier (pb_fast32.cuh): decision thresholds with guards sized for float
// arithmetic.  d: the unrounded constants (calibration reference); the kernels get the float copy.
// K (error bound = K * 2^-24 * shape) was calibrated with pb_debug_fast32_stats: see
// tests/test_gpu_parity.py::test_fp32_tier_error_bound for the ratios measured.
constexpr double kFast32K = 16.0;

static Fast32GeomT<double> derive_fast32(const OutGeom& o, const SrcGeom& s, const FastGeom& g) {
    Fast32GeomT<double> d;
    std::memset(&d, 0, sizeof(d));
    const double inf = INFINITY;
    d.enabled = g.enabled;
    if (const char* e = std::getenv("PB_FP32")) {
        if (std::atoi(e) == 0) d.enabled = 0;
    }
    // index32 keeps coordinates below 2^21; float pixel-centre coordinates must be exact
    if (o.H > (1 << 20) || o.W > (1 << 20) || s.H > (1 << 20) || s.W > (1 << 20)) d.enabled = 0;
    d.has_rot = g.has_rot;
    std::memcpy(d.rot, g.rot, sizeof(d.rot));
    d.r2_valid = d.r2_invalid = d.r2_domain = d.r2_nan = inf;
    if (o.kind == PB_KIND_EQUIRECT) {
        d.lon0 = o.x_start;
        d.lon_step = o.x_step;
        d.lat_step = o.y_step;
    } else {
        const double f = o.f, hf = o.half_fov, rel = 2e-5;
        d.x0 = o.x_start;
        d.y0 = o.y_start;
        d.inv_f = 1.0 / f;
        d.quarter_inv_f2 = 0.25 / (f * f);
        double d_star = inf;
        switch (o.lens) {
            case PB_LENS_EQUIDISTANT: d_star = hf; break;
            case PB_LENS_EQUISOLID: d_star = hf < kPi ? 2.0 * std::sin(hf / 2.0) : inf; break;
            case PB_LENS_ORTHOGRAPHIC: d_star = hf < kPi / 2 ? std::sin(hf) : inf; break;
            case PB_LENS_STEREOGRAPHIC: d_star = hf < kPi ? 2.0 * std::tan(hf / 2.0) : inf; break;
            case PB_LENS_RECTILINEAR: d_star = hf < kPi / 2 ? std::tan(hf) : inf; break;
            default: d_star = 0.713 * hf < kPi / 2 ? 1.47 * std::sin(0.713 * hf) : inf; break;
        }
        if (hf < 0.0) {
            d.r2_valid = d.r2_invalid = -1.0;
        } else if (d_star < inf) {
            const double r_star = d_star * f;
            d.r2_valid = (r_star * (1.0 - rel)) * (r_star * (1.0 - rel));
            d.r2_invalid = (r_star * (1.0 + rel)) * (r_star * (1.0 + rel));
        }
        // Lens inverses lose accuracy towards the edge of their domain (sqrt(1 - u) has a relative
        // error of eps / (2 (1 - u))): tier 1 stops where that amplification reaches ~4, the rest of
        // the image circle goes to the float64 tiers.  (Measured with the edge at 1 - 1e-3: error
        // ratios of 13 on a 360-degree equisolid output against 2-6 everywhere else.)
        switch (o.lens) {
            case PB_LENS_EQUISOLID: d.r2_domain = 4.0 * f * f * 0.88; break;      // lat < 139 deg
            case PB_LENS_ORTHOGRAPHIC: d.r2_domain = f * f * 0.94; break;          // lat < 76 deg
            case PB_LENS_THOBY: d.r2_domain = 1.47 * 1.47 * f * f * 0.94; break;
            case PB_LENS_EQUIDISTANT: d.r2_domain = (kPi * 0.999 * f) * (kPi * 0.999 * f); break;
            default: break;
        }
        // where asin() of the lens inverse leaves its domain (a NaN ray in the reference), with a guard
        switch (o.lens) {
            case PB_LENS_EQUISOLID: d.r2_nan = 4.0 * f * f * (1.0 - 1e-5); break;
            case PB_LENS_ORTHOGRAPHIC: d.r2_nan = f * f * (1.0 - 1e-5); break;
            case PB_LENS_THOBY: d.r2_nan = 1.47 * 1.47 * f * f * (1.0 - 1e-5); break;
            default: break;
        }
    }
    d.src_f = s.f;
    d.ny_band_lo = 2.0;
    d.ny_band_hi = -2.0;
    if (s.kind == PB_KIND_EQUIRECT) {
        d.inv_seg_h = 1.0 / s.seg_h;
        d.inv_seg_w = 1.0 / s.seg_w;
    } else {
        const double c = std::cos(s.rect_limit), guard = 1e-5;  // absolute guards on cos(lat)
        d.ny_rect_in = c + guard;
        d.ny_rect_out = c - guard;
        if (s.kind == PB_KIND_DOUBLE && s.mrg_lo <= s.mrg_hi_safe) {
            const double t_lo = std::fmin(s.mrg_lo, kPi - s.mrg_hi_safe);
            const double t_hi = std::fmax(s.mrg_hi_safe, kPi - s.mrg_lo);
            d.ny_band_hi = std::cos(std::fmax(t_lo, 0.0)) + guard;
            d.ny_band_lo = std::cos(std::fmin(t_hi, kPi)) - guard;
        }
    }
    double k = kFast32K;
    if (const char* e = std::getenv("PB_FP32_K")) k = std::atof(e);  // calibration experiments
    d.k_eps = k * 5.9604644775390625e-08;  // K * 2^-24
    return d;
}

// ------------------------------------------------------------------------------------ kernels

struct RemapArgs {
    OutGeom out;
    SrcGeom src;
    Rotations rot;
    FastGeom fast;
    const unsigned char* src_px;
    unsigned char* dst_px;
    long long src_frame_stride, dst_frame_stride;
    int n_frames;
    int row_begin, row_end;  // output rows this launch covers; dst_px points at row row_begin
};

// one pixel of C elements of T (uint8 images: T = unsigned char; wider elements: the unsigned
// integer of their width, so that the bytes move unconverted)
template <int C, typename T = unsigned char>
__device__ __forceinline__ void copy_px(T* __restrict__ d, const T* __restrict__ s) {
#pragma unroll
    for (int c = 0; c < C; ++c) d[c] = __ldg(s + c);
}

template <int C, typename T = unsigned char>
__device__ __forceinline__ void zero_px(T* __restrict__ d) {
#pragma unroll
    for (int c = 0; c < C; ++c) d[c] = 0;
}

// Generic fused remap: one thread resolves one output pixel (float64, every polar round trip
// of the reference kept), then applies the resolved lookup to every frame of the batch.
template <int OUT_KIND, int SRC_KIND, int C>
__global__ void __launch_bounds__(256) remap_generic_kernel(const __grid_constant__ RemapArgs a) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = a.row_begin + blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= a.row_end || j >= a.out.W) return;

    const Lookup L = resolve_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, i, j);
    const int off0 = xy_to_offset(L.xy0, a.src.W);
    const int off1 = xy_to_offset(L.xy1, a.src.W);

    const long long dst_off = ((long long)(i - a.row_begin) * a.out.W + j) * C;
    for (int f = 0; f < a.n_frames; ++f) {
        const unsigned char* __restrict__ sp = a.src_px + f * a.src_frame_stride;
        unsigned char* __restrict__ dp = a.dst_px + f * a.dst_frame_stride + dst_off;
        if (SRC_KIND != PB_KIND_DOUBLE) {
            if (off0 >= 0) copy_px<C>(dp, sp + (long long)off0 * C);
            else zero_px<C>(dp);
        } else {
            const unsigned char* p0 = sp + (long long)(off0 >= 0 ? off0 : 0) * C;
            const unsigned char* p1 = sp + (long long)(off1 >= 0 ? off1 : 0) * C;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const unsigned v0 = off0 >= 0 ? __ldg(p0 + c) : 0u;
                const unsigned v1 = off1 >= 0 ? __ldg(p1 + c) : 0u;
                dp[c] = blend_u8(v0, L.w0, v1, L.w1);
            }
        }
    }
}

// ONE frame, any geometry (rotated remaps above all): every thread resolves two quads of four
// consecutive pixels and gathers them straight from global memory -- no staging, no barrier.
// With a single frame the resolve (~150+ float64-heavy instructions per pixel even through the
// short cut) is all that matters: the tiled kernel's two-phase structure (resolve -> shared memory
// -> footprint -> TMA stage -> gather) costs ~85 instructions per pixel on top and buys nothing,
// because a warp's 32 byte-gathers of a smooth mapping touch only 8-12 sectors that mostly hit L1
// (measured: cfg2 153 -> 142 us even with the one-pixel-per-thread generic kernel).
// C = 3, W % 4 == 0, dst 4-byte aligned: a quad is 12 contiguous bytes = three aligned words.
#ifndef PB_DIRECT_MIN_CTAS
#define PB_DIRECT_MIN_CTAS 4
#endif
template <int OUT_KIND, int SRC_KIND>
__global__ void __launch_bounds__(256, PB_DIRECT_MIN_CTAS) remap_direct_kernel(const __grid_constant__ RemapArgs a) {
    constexpr bool DBL = (SRC_KIND == PB_KIND_DOUBLE);
    const int tid = threadIdx.x;
    const int j0 = blockIdx.x * kTileW + 4 * (tid & 7);
    if (j0 >= a.out.W) return;
    const unsigned char* __restrict__ sp = a.src_px;
    const int src_pitch = a.src.W * 3;
#pragma unroll 1
    for (int q = 0; q < 2; ++q) {
        const int i = a.row_begin + blockIdx.y * kTileH + (tid >> 3) + q * 32;
        if (i >= a.row_end) break;
        unsigned long long lo = 0;  // bytes 0..7 of the quad
        unsigned hi = 0;            // bytes 8..11
#pragma unroll 1
        for (int k = 0; k < 4; ++k) {
            const Lookup L = resolve_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, i, j0 + k);
            unsigned px = 0;
            if (L.xy0 >= 0) px = pick_px_global(sp, (L.xy0 >> 16) * src_pitch + (L.xy0 & 0xffff) * 3);
            if (DBL) {
                unsigned p1 = 0;
                if (L.xy1 >= 0) p1 = pick_px_global(sp, (L.xy1 >> 16) * src_pitch + (L.xy1 & 0xffff) * 3);
                px = blend_px(px, L.w0, p1, L.w1) & 0xffffffu;
            }
            const int sh = 24 * k;  // pixel k sits at bytes 3k .. 3k+2
            if (k < 3) lo |= (unsigned long long)px << sh;
            if (k == 2) hi |= px >> 16;
            if (k == 3) hi |= px << 8;
        }
        unsigned* o = reinterpret_cast<unsigned*>(a.dst_px + ((long long)(i - a.row_begin) * a.out.W + j0) * 3);
        o[0] = (unsigned)lo;
        o[1] = (unsigned)(lo >> 32);
        o[2] = hi;
    }
}

// The same for a camera / panorama source with the undecided pixels of a warp DEFERRED: every
// thread first runs tier 1 (float, pb_fast32.cuh) on its 8 pixels and parks the results in shared
// memory; the ~2 % of pixels tier 1 could not decide are then resolved through the float64 tiers.
// Run in place, two pixels in a hundred would put 1 - 0.98^32 = 48 % of the warps through the
// float64 code at every one of the 8 pixel steps, with one active lane each time.
#ifndef PB_DIRECT32_UNROLL
#define PB_DIRECT32_UNROLL 4
#endif
constexpr int kDirect32Unroll = PB_DIRECT32_UNROLL;
template <int OUT_KIND, int SRC_KIND>
__global__ void __launch_bounds__(256, PB_DIRECT_MIN_CTAS) remap_direct32_kernel(const __grid_constant__ RemapArgs a) {
    static_assert(SRC_KIND != PB_KIND_DOUBLE, "single-slot sources only");
    __shared__ int xybuf[8][kPxPerThread][32];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int row0 = a.row_begin + blockIdx.y * kTileH, col0 = blockIdx.x * kTileW;
    const int i0 = row0 + (tid >> 3), j0 = col0 + 4 * (tid & 7);
    unsigned pend = 0;  // bit p: tier 1 left pixel p of this thread undecided
    // the four pixels of a quad share their row: unrolled, so that what depends on the row alone is
    // computed once and four independent chains are in flight (PB_DIRECT32_UNROLL=1: one by one)
#pragma unroll 1
    for (int q = 0; q < kRowsPerThread; ++q) {
        const int i = i0 + q * 32;
#pragma unroll kDirect32Unroll
        for (int k = 0; k < 4; ++k) {
            const int p = q * 4 + k, j = j0 + k;
            int xy = kNoPixel;
            if (i < a.row_end && j < a.out.W) {
                Lookup L;
                if (a.fast.f32.enabled && fast32_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast.f32, a.src, i, j, L)) xy = L.xy0;
                else pend |= 1u << p;
            }
            xybuf[w][p][lane] = xy;
        }
    }
    // The undecided pixels -- a percent or two, spread evenly -- are taken AFTER the float passes,
    // every lane its own, one per round: a warp of 256 pixels has ~5 of them on ~5 different lanes,
    // so it goes through the float64 tiers once or twice instead of at almost every one of the 8
    // pixel steps (in place) -- and without the per-pixel ballot / queue bookkeeping a compacted
    // queue costs (measured: that bookkeeping is dearer than the second round it saves).
    while (__any_sync(0xffffffffu, pend != 0)) {
        if (pend) {
            const int p = __ffs(pend) - 1;
            pend &= pend - 1;
            const int i = i0 + (p >> 2) * 32, j = j0 + (p & 3);
            xybuf[w][p][lane] = resolve_lookup64<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, i, j).xy0;
        }
    }
    if (j0 >= a.out.W) return;
    const unsigned char* __restrict__ sp = a.src_px;
    const int src_pitch = a.src.W * 3;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int i = i0 + q * 32;
        if (i >= a.row_end) break;
        unsigned px[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int xy = xybuf[w][q * 4 + k][lane];
            px[k] = xy >= 0 ? pick_px_global(sp, (xy >> 16) * src_pitch + (xy & 0xffff) * 3) : 0u;
        }
        store_quad(reinterpret_cast<unsigned*>(a.dst_px + ((long long)(i - a.row_begin) * a.out.W + j0) * 3), px);
    }
}

// Calibration / self-check of tier 1 over every pixel of a geometry (pb_debug_fast32_stats):
// stats[0..1] = largest |float - double| / (2^-24 * shape) of a coordinate (x, y) as float bits,
// counters: [0] pixels, [1] undecided by tier 1, [2] decided by tier 1 but different from tiers 2/3,
// [3] float and double evaluations disagree on a pixel's status (fov / no-pixel decisions)
template <int OUT_KIND, int SRC_KIND>
__global__ void __launch_bounds__(256) fast32_stats_kernel(const __grid_constant__ RemapArgs a,
                                                           const __grid_constant__ Fast32GeomT<double> gd,
                                                           unsigned* __restrict__ maxima,
                                                           unsigned long long* __restrict__ counters) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= a.out.H || j >= a.out.W) return;
    const Coords32<float> cf = coords32<float, OUT_KIND, SRC_KIND>(a.out, a.fast.f32, a.src, i, j);
    const Coords32<double> cd = coords32<double, OUT_KIND, SRC_KIND>(a.out, gd, a.src, i, j);
    const double eps = 5.9604644775390625e-08;
    if (cf.status == 0 && cd.status == 0) {
        atomicMax(maxima + 0, __float_as_uint((float)(fabs((double)cf.vx - cd.vx) / (eps * (double)cf.ex))));
        atomicMax(maxima + 1, __float_as_uint((float)(fabs((double)cf.vy - cd.vy) / (eps * (double)cf.ey))));
    }
    if (SRC_KIND == PB_KIND_DOUBLE && cf.status != 2 && cd.status != 2 && cf.slot1 == 0 && cd.slot1 == 0) {
        atomicMax(maxima + 0, __float_as_uint((float)(fabs((double)cf.wx - cd.wx) / (eps * (double)cf.fx_))));
        atomicMax(maxima + 1, __float_as_uint((float)(fabs((double)cf.wy - cd.wy) / (eps * (double)cf.fy_))));
    }
    atomicAdd(counters + 0, 1ULL);
    if (cf.status != 2 && cd.status != 2 && (cf.status != cd.status || cf.slot1 != cd.slot1)) atomicAdd(counters + 3, 1ULL);
    Lookup L;
    if (!a.fast.f32.enabled || !fast32_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast.f32, a.src, i, j, L)) {
        atomicAdd(counters + 1, 1ULL);  // (a tier that is switched off decides nothing)
    } else {
        const Lookup R = resolve_lookup64<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, i, j);
        if (L.xy0 != R.xy0 || L.xy1 != R.xy1 || !(R.w0 == 1.0 && R.w1 == 1.0)) atomicAdd(counters + 2, 1ULL);
    }
}

// The calibration half of the above alone (pb_plan_create): largest |float - double| / (2^-24 * shape)
// of a coordinate over the pixels both evaluations give coordinates for, as float bits.
template <int OUT_KIND, int SRC_KIND>
__global__ void __launch_bounds__(256) fast32_ratio_kernel(const __grid_constant__ RemapArgs a,
                                                           const __grid_constant__ Fast32GeomT<double> gd,
                                                           unsigned* __restrict__ maxima) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    float r = 0.0f;
    if (i < a.out.H && j < a.out.W) {
        const Coords32<float> cf = coords32<float, OUT_KIND, SRC_KIND>(a.out, a.fast.f32, a.src, i, j);
        if (cf.status != 2) {
            const Coords32<double> cd = coords32<double, OUT_KIND, SRC_KIND>(a.out, gd, a.src, i, j);
            const double eps = 5.9604644775390625e-08;
            if (cf.status == 0 && cd.status == 0)
                r = fmaxf((float)(fabs((double)cf.vx - cd.vx) / (eps * (double)cf.ex)),
                          (float)(fabs((double)cf.vy - cd.vy) / (eps * (double)cf.ey)));
            if (SRC_KIND == PB_KIND_DOUBLE && cd.status != 2 && cf.slot1 == 0 && cd.slot1 == 0)
                r = fmaxf(r, fmaxf((float)(fabs((double)cf.wx - cd.wx) / (eps * (double)cf.fx_)),
                                   (float)(fabs((double)cf.wy - cd.wy) / (eps * (double)cf.fy_))));
            if (!(r >= 0.0f)) r = INFINITY;  // a NaN must not hide behind the maximum
        }
    }
    const unsigned bits = __reduce_max_sync(0xffffffffu, __float_as_uint(r));  // (non-negative floats order like their bits)
    if ((threadIdx.x & 31) == 0 && bits != 0) atomicMax(maxima, bits);
}

// get_coordinate_map() + n rotations, materialised.
template <int OUT_KIND>
__global__ void __launch_bounds__(256) materialize_map_kernel(const __grid_constant__ OutGeom out,
                                                              const __grid_constant__ Rotations rot,
                                                              double* __restrict__ map) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= out.H || j >= out.W) return;
    Ray r = output_ray<OUT_KIND>(out, i, j);
    for (int k = 0; k < rot.n; ++k) r = rotate_ray(r, rot.m[k]);
    double* m = map + ((long long)i * out.W + j) * 3;
    m[0] = r.lat;
    m[1] = r.lon;
    m[2] = r.invalid ? 1.0 : 0.0;
}

struct Mat3 {
    double m[9];
};

__global__ void __launch_bounds__(256) rotate_map_kernel(const __grid_constant__ Mat3 mat, double* __restrict__ in,
                                                         double* __restrict__ out, long long n) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    Ray r;
    r.lat = in[p * 3 + 0];
    r.lon = in[p * 3 + 1];
    r.invalid = in[p * 3 + 2] != 0.0;
    if (r.invalid) {  // rotation.py:124-125 zeroes the caller's map
        in[p * 3 + 0] = 0.0;
        in[p * 3 + 1] = 0.0;
    }
    r = rotate_ray(r, mat.m);
    out[p * 3 + 0] = r.lat;
    out[p * 3 + 1] = r.lon;
    out[p * 3 + 2] = r.invalid ? 1.0 : 0.0;
}

// T: one element of the image (unsigned char; for a camera / equirect source also the unsigned
// integer of a 2, 4 or 8-byte element -- the copy moves bytes, it converts nothing)
template <int SRC_KIND, int C, typename T = unsigned char>
__global__ void __launch_bounds__(256) gather_from_map_kernel(const __grid_constant__ SrcGeom src,
                                                              double* __restrict__ map, long long n,
                                                              const T* __restrict__ sp,
                                                              T* __restrict__ dst) {
    static_assert(SRC_KIND != PB_KIND_DOUBLE || sizeof(T) == 1, "the double-fisheye blend is uint8 arithmetic");
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    Ray r;
    r.lat = map[p * 3 + 0];
    r.lon = map[p * 3 + 1];
    r.invalid = map[p * 3 + 2] != 0.0;
    if (SRC_KIND == PB_KIND_EQUIRECT && r.invalid) {  // projection.py:533-536
        map[p * 3 + 0] = 0.0;
        map[p * 3 + 1] = 0.0;
    }
    const Lookup L = source_lookup<SRC_KIND>(src, r);
    const int off0 = xy_to_offset(L.xy0, src.W);
    const int off1 = xy_to_offset(L.xy1, src.W);
    T* dp = dst + p * C;
    if constexpr (SRC_KIND != PB_KIND_DOUBLE) {
        if (off0 >= 0) copy_px<C, T>(dp, sp + (long long)off0 * C);
        else zero_px<C, T>(dp);
    } else {
        if (r.invalid) {
            zero_px<C>(dp);
            return;
        }
        const unsigned char* p0 = sp + (long long)(off0 >= 0 ? off0 : 0) * C;
        const unsigned char* p1 = sp + (long long)(off1 >= 0 ? off1 : 0) * C;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const unsigned v0 = off0 >= 0 ? __ldg(p0 + c) : 0u;
            const unsigned v1 = off1 >= 0 ? __ldg(p1 + c) : 0u;
            dp[c] = blend_u8(v0, L.w0, v1, L.w1);
        }
    }
}

// map_projection (projection.py:550-599), a visualisation of a coordinate map: latitude -> red
// (stretched over the range it takes on the valid pixels), longitude -> green, invalid -> blue.
// Pass 1: smallest / largest latitude over the valid pixels (numpy.min / max: a NaN anywhere among
// them makes the result NaN) and, like the reference, (lat, lon) of the invalid pixels zeroed in
// place.  Doubles are compared through their order-preserving integer image.
__device__ __forceinline__ long long ordered_bits(double v) {
    const long long b = __double_as_longlong(v);
    return b < 0 ? (long long)(0x8000000000000000ULL - (unsigned long long)b) : b;
}
__device__ __forceinline__ double from_ordered_bits(long long o) {
    return __longlong_as_double(o < 0 ? (long long)(0x8000000000000000ULL - (unsigned long long)o) : o);
}
struct MapRange {
    long long lo, hi;  // ordered_bits of the smallest / largest valid latitude
    int any_nan, any_valid;
};
__global__ void __launch_bounds__(256) map_range_kernel(double* __restrict__ map, long long n, MapRange* __restrict__ range) {
    long long lo = 0x7fffffffffffffffLL, hi = (long long)0x8000000000000000ULL;
    int nan = 0, valid = 0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        if (map[p * 3 + 2] != 0.0) {  // projection.py:566: polar_map[invalid_map] = 0 (a view: the caller's map)
            map[p * 3 + 0] = 0.0;
            map[p * 3 + 1] = 0.0;
            continue;
        }
        const double lat = map[p * 3];
        valid = 1;
        if (lat != lat) nan = 1;
        else {
            const long long o = ordered_bits(lat);
            lo = o < lo ? o : lo;
            hi = o > hi ? o : hi;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const long long l2 = __shfl_xor_sync(0xffffffffu, lo, off), h2 = __shfl_xor_sync(0xffffffffu, hi, off);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
        nan |= __shfl_xor_sync(0xffffffffu, nan, off);
        valid |= __shfl_xor_sync(0xffffffffu, valid, off);
    }
    if ((threadIdx.x & 31) == 0) {
        if (valid) {
            atomicMin(&range->lo, lo);
            atomicMax(&range->hi, hi);
            atomicOr(&range->any_valid, 1);
        }
        if (nan) atomicOr(&range->any_nan, 1);
    }
}
__global__ void __launch_bounds__(256) map_projection_kernel(const double* __restrict__ map, long long n,
                                                             const MapRange* __restrict__ range, unsigned char* __restrict__ dst) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const double lo = range->any_nan ? nan : from_ordered_bits(range->lo);
    const double hi = range->any_nan ? nan : from_ordered_bits(range->hi);
    const double factor = __ddiv_rn(255.0, __dadd_rn(hi, -lo));  // :573-574
    const bool invalid = map[p * 3 + 2] != 0.0;
    double red = map[p * 3];
    if (!invalid) red = __dmul_rn(__dadd_rn(red, -lo), factor);  // :576-577 (two in-place passes: two roundings)
    const double green = __dmul_rn(255.0 / (kPi * 2), map[p * 3 + 1]);  // :583-584
    dst[p * 3 + 0] = cast_u8(rint(red));    // numpy.round: half to even
    dst[p * 3 + 1] = cast_u8(rint(green));
    dst[p * 3 + 2] = invalid ? 255 : 0;
}

// ------------------------------------------------------------------------------------ launchers

template <int OUT_KIND, int SRC_KIND>
static void launch_generic_c(const RemapArgs& a, cudaStream_t st) {
    dim3 block(32, 8);
    dim3 grid((a.out.W + block.x - 1) / block.x, (a.row_end - a.row_begin + block.y - 1) / block.y);
    switch (a.src.C) {
        case 1: remap_generic_kernel<OUT_KIND, SRC_KIND, 1><<<grid, block, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
        case 2: remap_generic_kernel<OUT_KIND, SRC_KIND, 2><<<grid, block, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
        case 3: remap_generic_kernel<OUT_KIND, SRC_KIND, 3><<<grid, block, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
        default: remap_generic_kernel<OUT_KIND, SRC_KIND, 4><<<grid, block, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
    }
}

template <int OUT_KIND>
static void launch_generic_s(const RemapArgs& a, cudaStream_t st) {
    switch (a.src.kind) {
        case PB_KIND_CAMERA: launch_generic_c<OUT_KIND, PB_KIND_CAMERA>(a, st); break;
        case PB_KIND_DOUBLE: launch_generic_c<OUT_KIND, PB_KIND_DOUBLE>(a, st); break;
        default: launch_generic_c<OUT_KIND, PB_KIND_EQUIRECT>(a, st); break;
    }
}

template <int OUT_KIND>
static void launch_direct_s(const RemapArgs& a, dim3 grid, cudaStream_t st) {
    switch (a.src.kind) {
        case PB_KIND_CAMERA: remap_direct_kernel<OUT_KIND, PB_KIND_CAMERA><<<grid, 256, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
        case PB_KIND_DOUBLE: remap_direct_kernel<OUT_KIND, PB_KIND_DOUBLE><<<grid, 256, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
        default: remap_direct_kernel<OUT_KIND, PB_KIND_EQUIRECT><<<grid, 256, 0, st>>>(a); PB_COUNT_LAUNCH(); break;
    }
}

template <int OUT_KIND>
static void launch_direct32_s(const RemapArgs& a, dim3 grid, cudaStream_t st) {
    if (a.src.kind == PB_KIND_CAMERA) remap_direct32_kernel<OUT_KIND, PB_KIND_CAMERA><<<grid, 256, 0, st>>>(a);
    else remap_direct32_kernel<OUT_KIND, PB_KIND_EQUIRECT><<<grid, 256, 0, st>>>(a);
    PB_COUNT_LAUNCH();
}

template <int OUT_KIND>
static void launch_stats_s(const RemapArgs& a, const Fast32GeomT<double>& gd, unsigned* maxima, unsigned long long* counters,
                           cudaStream_t st) {
    dim3 block(32, 8);
    dim3 grid((a.out.W + 31) / 32, (a.out.H + 7) / 8);
    switch (a.src.kind) {
        case PB_KIND_CAMERA: fast32_stats_kernel<OUT_KIND, PB_KIND_CAMERA><<<grid, block, 0, st>>>(a, gd, maxima, counters); break;
        case PB_KIND_DOUBLE: fast32_stats_kernel<OUT_KIND, PB_KIND_DOUBLE><<<grid, block, 0, st>>>(a, gd, maxima, counters); break;
        default: fast32_stats_kernel<OUT_KIND, PB_KIND_EQUIRECT><<<grid, block, 0, st>>>(a, gd, maxima, counters); break;
    }
    PB_COUNT_LAUNCH();
}

template <int OUT_KIND>
static void launch_ratio_s(const RemapArgs& a, const Fast32GeomT<double>& gd, unsigned* maxima, cudaStream_t st) {
    dim3 block(32, 8);
    dim3 grid((a.out.W + block.x - 1) / block.x, (a.out.H + block.y - 1) / block.y);
    switch (a.src.kind) {
        case PB_KIND_CAMERA: fast32_ratio_kernel<OUT_KIND, PB_KIND_CAMERA><<<grid, block, 0, st>>>(a, gd, maxima); break;
        case PB_KIND_DOUBLE: fast32_ratio_kernel<OUT_KIND, PB_KIND_DOUBLE><<<grid, block, 0, st>>>(a, gd, maxima); break;
        default: fast32_ratio_kernel<OUT_KIND, PB_KIND_EQUIRECT><<<grid, block, 0, st>>>(a, gd, maxima); break;
    }
    PB_COUNT_LAUNCH();
}

static void launch_direct(const RemapArgs& a, cudaStream_t st) {
    dim3 grid((a.out.W + kTileW - 1) / kTileW, (a.row_end - a.row_begin + kTileH - 1) / kTileH);
    static const bool compact_off = std::getenv("PB_COMPACT") && std::atoi(std::getenv("PB_COMPACT")) == 0;  // experiments
    if (a.src.kind != PB_KIND_DOUBLE && a.fast.f32.enabled && !compact_off) {
        switch (a.out.kind) {
            case PB_KIND_CAMERA: launch_direct32_s<PB_KIND_CAMERA>(a, grid, st); break;
            case PB_KIND_DOUBLE: launch_direct32_s<PB_KIND_DOUBLE>(a, grid, st); break;
            default: launch_direct32_s<PB_KIND_EQUIRECT>(a, grid, st); break;
        }
        return;
    }
    switch (a.out.kind) {
        case PB_KIND_CAMERA: launch_direct_s<PB_KIND_CAMERA>(a, grid, st); break;
        case PB_KIND_DOUBLE: launch_direct_s<PB_KIND_DOUBLE>(a, grid, st); break;
        default: launch_direct_s<PB_KIND_EQUIRECT>(a, grid, st); break;
    }
}

static void launch_generic(const RemapArgs& a, cudaStream_t st) {
    switch (a.out.kind) {
        case PB_KIND_CAMERA: launch_generic_s<PB_KIND_CAMERA>(a, st); break;
        case PB_KIND_DOUBLE: launch_generic_s<PB_KIND_DOUBLE>(a, st); break;
        default: launch_generic_s<PB_KIND_EQUIRECT>(a, st); break;
    }
}

template <int SRC_KIND>
static void launch_gather_c(const SrcGeom& s, double* map, long long n, const unsigned char* sp,
                            unsigned char* dst, cudaStream_t st) {
    const int block = 256;
    const unsigned grid = (unsigned)((n + block - 1) / block);
    switch (s.C) {
        case 1: gather_from_map_kernel<SRC_KIND, 1><<<grid, block, 0, st>>>(s, map, n, sp, dst); PB_COUNT_LAUNCH(); break;
        case 2: gather_from_map_kernel<SRC_KIND, 2><<<grid, block, 0, st>>>(s, map, n, sp, dst); PB_COUNT_LAUNCH(); break;
        case 3: gather_from_map_kernel<SRC_KIND, 3><<<grid, block, 0, st>>>(s, map, n, sp, dst); PB_COUNT_LAUNCH(); break;
        default: gather_from_map_kernel<SRC_KIND, 4><<<grid, block, 0, st>>>(s, map, n, sp, dst); PB_COUNT_LAUNCH(); break;
    }
}

// the same for elements of T (2, 4 or 8 bytes), camera / equirect sources
template <int SRC_KIND, typename T>
static void launch_gather_wide(const SrcGeom& s, double* map, long long n, const void* src, void* dst, cudaStream_t st) {
    const int block = 256;
    const unsigned grid = (unsigned)((n + block - 1) / block);
    const T* sp = static_cast<const T*>(src);
    T* dp = static_cast<T*>(dst);
    switch (s.C) {
        case 1: gather_from_map_kernel<SRC_KIND, 1, T><<<grid, block, 0, st>>>(s, map, n, sp, dp); break;
        case 2: gather_from_map_kernel<SRC_KIND, 2, T><<<grid, block, 0, st>>>(s, map, n, sp, dp); break;
        case 3: gather_from_map_kernel<SRC_KIND, 3, T><<<grid, block, 0, st>>>(s, map, n, sp, dp); break;
        default: gather_from_map_kernel<SRC_KIND, 4, T><<<grid, block, 0, st>>>(s, map, n, sp, dp); break;
    }
    PB_COUNT_LAUNCH();
}

template <int SRC_KIND>
static void launch_gather_e(const SrcGeom& s, int elem_bytes, double* map, long long n, const void* src, void* dst,
                            cudaStream_t st) {
    switch (elem_bytes) {
        case 2: launch_gather_wide<SRC_KIND, unsigned short>(s, map, n, src, dst, st); break;
        case 4: launch_gather_wide<SRC_KIND, unsigned>(s, map, n, src, dst, st); break;
        default: launch_gather_wide<SRC_KIND, unsigned long long>(s, map, n, src, dst, st); break;
    }
}

// fused remap of pixels wider than one byte (pb_wide.cuh): VEC-byte words
template <int OUT_KIND, int SRC_KIND, bool SEP>
static void launch_wide_v(const WideArgs& a, int vec, dim3 grid, cudaStream_t st) {
    switch (vec) {
        case 16: remap_wide_kernel<OUT_KIND, SRC_KIND, SEP, 16><<<grid, 256, 0, st>>>(a); break;
        case 8: remap_wide_kernel<OUT_KIND, SRC_KIND, SEP, 8><<<grid, 256, 0, st>>>(a); break;
        case 4: remap_wide_kernel<OUT_KIND, SRC_KIND, SEP, 4><<<grid, 256, 0, st>>>(a); break;
        default: remap_wide_kernel<OUT_KIND, SRC_KIND, SEP, 2><<<grid, 256, 0, st>>>(a); break;
    }
    PB_COUNT_LAUNCH();
}

template <int OUT_KIND>
static void launch_wide_s(const WideArgs& a, int vec, dim3 grid, cudaStream_t st) {
    if (a.src.kind == PB_KIND_CAMERA) launch_wide_v<OUT_KIND, PB_KIND_CAMERA, false>(a, vec, grid, st);
    else launch_wide_v<OUT_KIND, PB_KIND_EQUIRECT, false>(a, vec, grid, st);
}

// The widest word (a power of two, at most 16 bytes) that divides the pixel size and every address
// the gather forms: the base pointers, and the frame strides when there is more than one frame
// (row pitches are whole pixels).
static int wide_vec(int px_bytes, const void* src, const void* dst, long long src_stride, long long dst_stride,
                    bool multi) {
    unsigned long long bits = (unsigned long long)px_bytes | (unsigned long long)reinterpret_cast<uintptr_t>(src) |
                              (unsigned long long)reinterpret_cast<uintptr_t>(dst);
    if (multi) bits |= (unsigned long long)src_stride | (unsigned long long)dst_stride;
    int vec = 16;
    while (vec > 2 && (bits & (unsigned long long)(vec - 1)) != 0) vec >>= 1;
    return vec;
}

// ------------------------------------------------------------------------------------ tiled path

// cuTensorMapEncodeTiled, fetched through the runtime so that libcuda is not a link dependency
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            (void)cudaGetLastError();
    }
    return fn;
}

// 3-D map over a batch of HWC uint8 frames seen as rows of bytes: {row bytes, rows, frames}
static bool encode_frames_map(CUtensorMap* map, const void* base, long long pitch, int rows, int frames,
                              long long frame_stride, int elem_bytes, int box_bytes, int box_rows) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)(pitch / elem_bytes), (cuuint64_t)rows, (cuuint64_t)frames};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)(frames > 1 ? frame_stride : pitch * rows)};
    const cuuint32_t box[3] = {(cuuint32_t)(box_bytes / elem_bytes), (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8;
    return enc(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int kMaxTiledSmem = 200 * 1024;
constexpr int kMaxDevices = 64;

template <int OUT_KIND, int SRC_KIND, int MODE, int CLS = 0>
static cudaError_t launch_tiled_one(const TiledArgs& a, cudaStream_t st) {
    const int smem = tiled_smem_bytes<SRC_KIND, MODE>(a.stage_bytes, a.n_buffers, a.n_out);
    // per instantiation and per device: the attribute belongs to the function on one device
    static bool configured[kMaxDevices] = {false};
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev)) return e;
    if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(remap_tiled_kernel<OUT_KIND, SRC_KIND, MODE, CLS>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxTiledSmem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
    }
    const int grid = a.tile_list ? a.n_list : a.tiles_x * a.tiles_y;
    if (grid <= 0) return cudaSuccess;
    remap_tiled_kernel<OUT_KIND, SRC_KIND, MODE, CLS><<<grid, kTileThreads, smem, st>>>(a);
    PB_COUNT_LAUNCH();
    return cudaGetLastError();
}

template <int OUT_KIND>
static cudaError_t launch_tiled_generic_s(const TiledArgs& a, cudaStream_t st) {
    switch (a.src.kind) {
        case PB_KIND_CAMERA: return launch_tiled_one<OUT_KIND, PB_KIND_CAMERA, 0>(a, st);
        case PB_KIND_DOUBLE: return launch_tiled_one<OUT_KIND, PB_KIND_DOUBLE, 0>(a, st);
        default: return launch_tiled_one<OUT_KIND, PB_KIND_EQUIRECT, 0>(a, st);
    }
}

static cudaError_t launch_tiled(const TiledArgs& a, bool separable, cudaStream_t st) {
    if (separable) {
        if (a.src.kind == PB_KIND_CAMERA) return launch_tiled_one<PB_KIND_EQUIRECT, PB_KIND_CAMERA, 1>(a, st);
        return launch_tiled_one<PB_KIND_EQUIRECT, PB_KIND_DOUBLE, 1>(a, st);
    }
    switch (a.out.kind) {
        case PB_KIND_CAMERA: return launch_tiled_generic_s<PB_KIND_CAMERA>(a, st);
        case PB_KIND_DOUBLE: return launch_tiled_generic_s<PB_KIND_DOUBLE>(a, st);
        default: return launch_tiled_generic_s<PB_KIND_EQUIRECT>(a, st);
    }
}

// batches with the source staged as a chunk list (pb_chunk.cuh)
template <int SRC_KIND, int CLS>
static cudaError_t launch_chunk_one(const TiledArgs& a, cudaStream_t st) {
    const int smem = chunk_smem_bytes(a.stage_bytes);
    static int max_smem_set[kMaxDevices] = {0};
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev)) return e;
    if (dev < 0 || dev >= kMaxDevices || smem > max_smem_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(remap_chunk_kernel<SRC_KIND, CLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kMaxDevices) max_smem_set[dev] = smem;
    }
    const int grid = a.tile_list ? a.n_list : a.tiles_x * a.tiles_y;
    if (grid <= 0) return cudaSuccess;
    remap_chunk_kernel<SRC_KIND, CLS><<<grid, kTileThreads, smem, st>>>(a);
    PB_COUNT_LAUNCH();
    return cudaGetLastError();
}

// the two-lens / blend-band class of a batch with 512 threads per CTA (pb_tiled2.cuh)
static cudaError_t launch_two_lens(const TiledArgs& a, cudaStream_t st) {
    const int smem = two_lens_smem_bytes(a.stage_bytes);
    static int max_smem_set[kMaxDevices] = {0};
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev)) return e;
    if (dev < 0 || dev >= kMaxDevices || smem > max_smem_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(remap_two_lens_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kMaxDevices) max_smem_set[dev] = smem;
    }
    if (a.n_list <= 0) return cudaSuccess;
    remap_two_lens_kernel<<<a.n_list, kTile2Threads, smem, st>>>(a);
    PB_COUNT_LAUNCH();
    return cudaGetLastError();
}

// tuning experiments
static int env_int(const char* name, int fallback) {
    const char* e = std::getenv(name);
    return e ? std::atoi(e) : fallback;
}
static bool class_split_off() { return env_int("PB_CLASS_SPLIT", 1) == 0; }

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// persistent single-frame kernel: as many CTAs as the device holds at once
template <int SRC_KIND, int NB, int CLS = 0>
static cudaError_t launch_sep1_one(const TiledArgs& a, cudaStream_t st) {
    const int smem = sep1_smem_bytes(a.sep1_cap, SRC_KIND == PB_KIND_DOUBLE, NB);
    static int max_smem_set[kMaxDevices] = {0};  // per device: the attribute belongs to the function on one device
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices || smem > max_smem_set[dev]) {
        e = cudaFuncSetAttribute(remap_sep1_kernel<SRC_KIND, NB, CLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < kMaxDevices) max_smem_set[dev] = smem;
    }
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, remap_sep1_kernel<SRC_KIND, NB, CLS>, kTileThreads, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    int grid = sms * per_sm;
    if (const char* env = std::getenv("PB_SEP1_WAVES")) grid *= std::atoi(env);  // tuning experiments
    if (const char* env = std::getenv("PB_SEP1_GRID")) grid = std::atoi(env);
    const int n_tiles = a.tile_list ? a.n_list : a.tiles_x * a.tiles_y;
    if (n_tiles <= 0) return cudaSuccess;
    if (grid > n_tiles) grid = n_tiles;
    if (grid < 1) grid = 1;
    // launched with programmatic stream serialisation: the prologue of this grid may overlap the
    // tail of the one before it on the stream (the kernel waits, griddepcontrol.wait, before it
    // touches an image): back to back cfg1 x1 25.6 -> 24.8 us, T x1 38.2 -> 38.0 us; the two grids
    // of a double-fisheye source lose 1.5 % with it and are launched plainly.  PB_PDL=0: plain launch
    static const bool pdl = env_int("PB_PDL", 1) != 0 && SRC_KIND == PB_KIND_CAMERA;
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kTileThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl ? 1 : 0;
    e = cudaLaunchKernelEx(&cfg, remap_sep1_kernel<SRC_KIND, NB, CLS>, a);
    PB_COUNT_LAUNCH();
    return e;
}

}  // namespace pb

// A plan: one validated geometry with everything derived from it (host constants, and for an
// un-rotated equirect output the separable device tables).
struct pb_plan {
    pb_remap_desc desc;
    pb::OutGeom out;
    pb::SrcGeom src;
    pb::Rotations rot;
    pb::FastGeom fast;   // thresholds of the guarded short cut (pb_fast.cuh)
    bool separable;      // un-rotated equirect output, camera / double source
    int stage_bytes;     // capacity of one stage buffer (a tile stages rows x its own row pitch)
    int max_units;       // widest staged row of any tile, in 16-byte units (one tensor map per width)
    int raster_band;     // tile rows per raster band (see remap_tiled_kernel)
    int sep1_cap;        // single-frame separable kernel: bytes per stage buffer
    int sep1_cap3;       // ... single-lens source: buffer size at which THREE stage buffers keep four CTAs per SM
                         //     and still hold (all but 3 % of) the tiles; 0 = two buffers
    double* luts;        // device: lens tables of PB_LENS_TABLE lenses (out.lut / src.lut point into it); null otherwise
    double* tables;      // device: col_tab [W][2], row_tab [H][4], then the per-tile footprints; null unless separable
    // separable double-fisheye source: the tiles sorted into two classes, each in raster order --
    // [0, n_one): exactly one lens visible at unit weights, [n_one, n_one + n_rest): the rest
    // (both lenses, blend band, nothing visible); batches run them as two launches (remap_tiled_kernel CLS)
    int* tile_lists;
    int n_one, n_rest;
    int4* sep1_cls;      // single-frame kernel: descriptor tables of the two classes ([n_one] then [n_rest][2])
    int sep1_cap_one;    // ... and the stage-buffer capacity of the one-lens class
    // the two grids of a double-fisheye remap are independent (disjoint tiles): the second one is
    // forked onto a stream of the plan's own and joined back, so that it fills the SMs the first
    // one's last wave leaves idle.  A few lanes (side stream + event pair), one per caller stream
    // seen, so that the frames of a pipeline that cycles over several streams do not serialise on
    // one side stream.
    static constexpr int kSideLanes = 4;
    struct SideLane {
        cudaStream_t side;
        cudaEvent_t ev_fork, ev_join;
        cudaStream_t user;  // caller stream this lane last served
    } lanes[kSideLanes];
    int n_lanes, next_lane;
    int device;
    // Encoded tensor maps, by buffer: a pipeline that cycles over a few device buffers pays
    // cuTensorMapEncodeTiled once per buffer instead of up to 15 times per launch (host latency on
    // a 40-60 us kernel).  A map only holds the address and the extents, so an entry stays valid
    // for whatever lives at that address later.
    static constexpr int kMapSlots = 8;
    struct SrcMaps {
        const void* base;
        long long stride;
        int frames, units;
        unsigned long long tick;
        CUtensorMap maps[pb::kMaxSrcMaps];
    } src_cache[kMapSlots];
    struct DstMap {
        const void* base;
        long long stride;
        int frames, rows;
        unsigned long long tick;
        CUtensorMap map;
    } dst_cache[kMapSlots];
    unsigned long long tick;
    double fast32_k;      // K of the FP32-first tier's error bound for this plan (calibrate_fast32; 16 un-calibrated)
    float fast32_ratio;   // what the calibration measured (-1: not run)
    // launches through one plan are serialised on the host (map caches, side lanes): a plan may be
    // shared by host threads
    std::mutex mu;
};

namespace pb {

static int validate_desc(const pb_remap_desc* desc, const char* who) {
    if (!desc) return fail(PB_ERR_INVALID_ARGUMENT, std::string(who) + ": null descriptor");
    if (int rc = check_image(desc->out, "out")) return rc;
    if (int rc = check_image(desc->src, "src")) return rc;
    if (desc->src.height > 32767 || desc->src.width > 65535)
        return fail(PB_ERR_UNSUPPORTED, std::string(who) + ": source larger than 32767 rows x 65535 columns");
    if (desc->channels < 1 || desc->channels > 4)
        return fail(PB_ERR_UNSUPPORTED, std::string(who) + ": channels must be 1..4");
    if (desc->n_rotations < 0) return fail(PB_ERR_INVALID_ARGUMENT, std::string(who) + ": negative n_rotations");
    if (desc->n_rotations > PB_MAX_ROTATIONS)
        return fail(PB_ERR_TOO_MANY_ROTATIONS, std::string(who) + ": more than PB_MAX_ROTATIONS rotations");
    return PB_OK;
}

static void plan_init(pb_plan& p, const pb_remap_desc& d) {
    p.desc = d;
    p.out = derive_out(d.out);
    p.src = derive_src(d.src, d.channels);
    p.rot.n = d.n_rotations;
    std::memcpy(p.rot.m, d.rotations, sizeof(p.rot.m));
    p.fast = derive_fast(d.out, p.out, d.src, p.src, d.n_rotations, d.rotations);
    p.fast.f32 = fast32_to_float(derive_fast32(p.out, p.src, p.fast));
    p.fast32_k = kFast32K;
    p.fast32_ratio = -1.0f;
    p.separable = d.out.kind == PB_KIND_EQUIRECT && d.n_rotations == 0 && d.src.kind != PB_KIND_EQUIRECT &&
                  d.channels == 3;
    p.stage_bytes = 24 * 1024;  // un-tuned default (pb_remap_u8 without a plan)
    p.max_units = 19;           // rows of up to 304 bytes = 101 source pixels
    p.raster_band = 16;
    p.sep1_cap = (d.src.kind == PB_KIND_DOUBLE ? 48 : 24) * 1024;  // un-tuned default
    p.sep1_cap3 = 0;
    if (const char* e = std::getenv("PB_RASTER_BAND")) p.raster_band = std::atoi(e);  // tuning experiments
    p.luts = nullptr;
    p.tables = nullptr;
    p.tile_lists = nullptr;
    p.n_one = p.n_rest = 0;
    p.sep1_cls = nullptr;
    p.sep1_cap_one = 24 * 1024;
    std::memset(p.lanes, 0, sizeof(p.lanes));
    p.n_lanes = p.next_lane = 0;
    p.device = -1;
    std::memset(p.src_cache, 0, sizeof(p.src_cache));
    std::memset(p.dst_cache, 0, sizeof(p.dst_cache));
    p.tick = 0;
}

// Footprint census of a geometry (one probe launch of the tiled kernel, nothing is remapped):
// picks the smallest staged-row width and box count that hold the footprint of ~all tiles, so that
// the stage buffers are as small -- and the occupancy as high -- as this geometry allows.
static int tiles_x(const pb_plan& p) { return (p.out.W + kTileW - 1) / kTileW; }
static int tiles_y(const pb_plan& p) { return (p.out.H + kTileH - 1) / kTileH; }
static int footprint_entries(const pb_plan& p) {
    return tiles_x(p) * tiles_y(p) * (p.src.kind == PB_KIND_DOUBLE ? 2 : 1);
}
// col_tab [W][2] + row_tab [H][4] doubles, then one int4 footprint per (tile, slot), then the same
// per (tile in launch order, slot) for the single-frame kernel
static size_t sep1_row_doubles(const pb_plan& p) { return p.src.kind == PB_KIND_DOUBLE ? 4 : 1; }
static size_t table_doubles(const pb_plan& p) {
    return 2 * (size_t)p.out.W + 4 * (size_t)p.out.H + 4 * (size_t)footprint_entries(p) +
           2 * (size_t)tiles_x(p) * kTileW + sep1_row_doubles(p) * (size_t)tiles_y(p) * kTileH;
}
static const int4* sep1_table(const pb_plan& p, const double* tables) {
    return reinterpret_cast<const int4*>(tables + 2 * (size_t)p.out.W + 4 * (size_t)p.out.H) + footprint_entries(p);
}
// (W and H need not be even: the int4 tables keep everything after them 16-byte aligned only if
// 2W + 4H is even, which it is)
static const double* sep1_col(const pb_plan& p, const double* tables) {
    return tables + 2 * (size_t)p.out.W + 4 * (size_t)p.out.H + 4 * (size_t)footprint_entries(p);
}
static const double* sep1_row(const pb_plan& p, const double* tables) {
    return sep1_col(p, tables) + 2 * (size_t)tiles_x(p) * kTileW;
}
static const int4* footprint_table(const pb_plan& p, const double* tables) {
    return reinterpret_cast<const int4*>(tables + 2 * (size_t)p.out.W + 4 * (size_t)p.out.H);
}

// Picks the stage-buffer capacity from the census h (see kProbeSizeBins): the smallest size that
// holds the footprint of all but 0.5 % of the (tile, slot) items -- the rest gather straight from
// global memory -- so that the buffers are as small, and the occupancy as high, as the geometry
// allows.  Staged rows are an odd number of 16-byte units wide (stage_units): vertically adjacent
// source pixels then sit 4*odd banks apart (8 distinct bank groups) instead of piling onto 1-4 of
// them, which is what the gather of a tile whose footprint runs down the source image would
// otherwise do (tests/analysis/stage_sim.py: 4.4 -> 2.3 wavefronts per LDS at pitch 256 -> 272).
static void pick_stage(pb_plan& p, const int* h) {
    long long items = 0;
    for (int k = 0; k < kProbeSizeBins; ++k) items += h[k];
    if (items <= 0) return;
    const long long need = items - items / 200;
    long long acc = 0;
    int kib = kProbeSizeBins - 1;
    for (int k = 0; k < kProbeSizeBins; ++k) {
        acc += h[k];
        if (acc >= need) { kib = k; break; }
    }
    if (kib < 2) kib = 2;
    if (kib > 48) kib = 48;
    if (const char* e = std::getenv("PB_STAGE_KIB")) kib = std::atoi(e);  // tuning experiments
    p.stage_bytes = kib * 1024;
    int units = h[kProbeSizeBins];
    if (units < kMinStageUnits) units = kMinStageUnits;
    if (units > kMaxStageUnits) units = kMaxStageUnits;
    p.max_units = units | 1;
}

// Double-fisheye source: which tiles see exactly one lens at unit blend weights (same test as the
// kernel's: the 64 rows of the tile, rows past the image edge repeating the last one), in the
// order the kernel rasters them.  fp: the plan's footprints on the host.
static void classify_tiles(pb_plan& p, const int4* fp, cudaStream_t st) {
    if (p.src.kind != PB_KIND_DOUBLE || p.tile_lists) return;
    const int tx = tiles_x(p), ty = tiles_y(p), n_tiles = tx * ty, H = p.out.H;
    std::vector<double> rows(4 * (size_t)H);
    if (cudaMemcpyAsync(rows.data(), p.tables + 2 * (size_t)p.out.W, rows.size() * sizeof(double), cudaMemcpyDeviceToHost,
                        st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    std::vector<char> unit_rows(ty);  // every row of the tile row has both weights exactly 1
    for (int t = 0; t < ty; ++t) {
        bool unit = true;
        for (int r = t * kTileH; r < (t + 1) * kTileH; ++r) {
            const int i = r < H ? r : H - 1;
            unit = unit && rows[4 * (size_t)i + 2] == 1.0 && rows[4 * (size_t)i + 3] == 1.0;
        }
        unit_rows[t] = unit;
    }
    std::vector<int> one, rest;
    for (int b = 0; b < n_tiles; ++b) {
        int x, y;
        if (p.raster_band > 0) {  // as remap_tiled_kernel walks them
            const int per_band = p.raster_band * tx, band = b / per_band, within = b - band * per_band;
            const int bh = std::min(p.raster_band, ty - band * p.raster_band);
            x = within / bh;
            y = band * p.raster_band + (within - x * bh);
        } else {
            y = b / tx;
            x = b - y * tx;
        }
        const int t = y * tx + x;
        const bool l = fp[2 * t].z > 0, r = fp[2 * t + 1].z > 0;
        ((l != r) && unit_rows[y] ? one : rest).push_back(t);
    }
    int* lists = nullptr;
    if (cudaMalloc((void**)&lists, sizeof(int) * n_tiles) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    one.insert(one.end(), rest.begin(), rest.end());
    if (cudaMemcpyAsync(lists, one.data(), sizeof(int) * n_tiles, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        (void)cudaGetLastError();
        cudaFree(lists);
        return;
    }
    p.tile_lists = lists;
    p.n_rest = (int)rest.size();
    p.n_one = n_tiles - p.n_rest;
    // single-frame kernel: per-class descriptor tables, and a buffer size that holds the one
    // rectangle of (all but 0.5 % of) the one-lens tiles
    int4* cls = nullptr;
    if (cudaMalloc((void**)&cls, sizeof(int4) * ((size_t)p.n_one + 2 * (size_t)p.n_rest + 1)) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    if (p.n_one > 0)
        pb_sep1_table_kernel<<<(p.n_one + 255) / 256, 256, 0, st>>>(footprint_table(p, p.tables), cls, tx, ty, p.raster_band,
                                                                   2, lists, p.n_one, 1);
    if (p.n_rest > 0)
        pb_sep1_table_kernel<<<(p.n_rest + 255) / 256, 256, 0, st>>>(footprint_table(p, p.tables), cls + p.n_one, tx, ty,
                                                                    p.raster_band, 2, lists + p.n_one, p.n_rest, 0);
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
        (void)cudaGetLastError();
        cudaFree(cls);
        return;
    }
    std::vector<int> kib;
    for (int i = 0; i < p.n_one; ++i) {
        const int t = one[i];
        const int4& f = fp[2 * t].z > 0 ? fp[2 * t] : fp[2 * t + 1];
        const int units = stage_units(f.w >> 1);
        kib.push_back(units <= kMaxStageUnits ? (f.z * kBoxRows * 16 * units + 1023) >> 10 : 1 << 20);
    }
    if (!kib.empty()) {
        std::sort(kib.begin(), kib.end());
        int k = kib[kib.size() - 1 - kib.size() / 200];
        p.sep1_cap_one = std::min(std::max(k, 4), 96) * 1024;
    }
    p.sep1_cls = cls;
    // the side stream carries the latency-bound grid (two-lens tiles) at the highest priority: its
    // CTAs are dispatched first wherever an SM has room, so they mix with the bandwidth-bound
    // one-lens CTAs over the whole run instead of queueing behind them (cfg5 x16 0.634 -> 0.620 ms)
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    for (int k = 0; k < pb_plan::kSideLanes; ++k) {
        pb_plan::SideLane& l = p.lanes[k];
        if (cudaStreamCreateWithPriority(&l.side, cudaStreamNonBlocking, env_int("PB_SIDE_PRIO", 1) ? prio_hi : prio_lo) != cudaSuccess ||
            cudaEventCreateWithFlags(&l.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&l.ev_join, cudaEventDisableTiming) != cudaSuccess) {
            (void)cudaGetLastError();
            if (l.side) cudaStreamDestroy(l.side);
            if (l.ev_fork) cudaEventDestroy(l.ev_fork);
            if (l.ev_join) cudaEventDestroy(l.ev_join);
            std::memset(&l, 0, sizeof(l));
            break;
        }
        p.n_lanes = k + 1;
    }
}

// fork: a side stream of the plan picks up after everything enqueued on st so far; join: st waits
// for it.  The lane is the one that served this caller stream last, else the next in turn.
// (called with the plan's mutex held)
static pb_plan::SideLane* fork_side(pb_plan& p, cudaStream_t st) {
    if (p.n_lanes == 0 || env_int("PB_CONCURRENT", 1) == 0) return nullptr;
    pb_plan::SideLane* l = nullptr;
    for (int k = 0; k < p.n_lanes; ++k)
        if (p.lanes[k].user == st) l = &p.lanes[k];
    if (!l) {
        l = &p.lanes[p.next_lane];
        p.next_lane = (p.next_lane + 1) % p.n_lanes;
        l->user = st;
    }
    if (cudaEventRecord(l->ev_fork, st) != cudaSuccess || cudaStreamWaitEvent(l->side, l->ev_fork, 0) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return l;
}
static cudaError_t join_side(pb_plan::SideLane* l, cudaStream_t st) {
    if (!l) return cudaSuccess;
    cudaError_t e = cudaEventRecord(l->ev_join, l->side);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(st, l->ev_join, 0);
    return e;
}

// The plan's tensor maps for these buffers, encoded on first use (called with the mutex held).
static bool cached_src_maps(pb_plan& p, const void* src, long long src_pitch, int frames, long long stride, int units,
                            CUtensorMap* out) {
    pb_plan::SrcMaps* hit = nullptr;
    pb_plan::SrcMaps* victim = &p.src_cache[0];
    for (auto& e : p.src_cache) {
        if (e.tick && e.base == src && e.stride == stride && e.frames == frames && e.units == units) hit = &e;
        if (e.tick < victim->tick) victim = &e;
    }
    if (!hit) {
        hit = victim;
        hit->tick = 0;
        for (int u = kMinStageUnits; u <= units; u += 2)
            if (!encode_frames_map(&hit->maps[(u - kMinStageUnits) / 2], src, src_pitch, p.src.H, frames, stride, 2, 16 * u,
                                   kBoxRows))
                return false;
        hit->base = src;
        hit->stride = stride;
        hit->frames = frames;
        hit->units = units;
    }
    hit->tick = ++p.tick;
    std::memcpy(out, hit->maps, sizeof(hit->maps));
    return true;
}
static bool cached_dst_map(pb_plan& p, const void* dst, long long dst_pitch, int rows, int frames, long long stride,
                           CUtensorMap* out) {
    pb_plan::DstMap* hit = nullptr;
    pb_plan::DstMap* victim = &p.dst_cache[0];
    for (auto& e : p.dst_cache) {
        if (e.tick && e.base == dst && e.stride == stride && e.frames == frames && e.rows == rows) hit = &e;
        if (e.tick < victim->tick) victim = &e;
    }
    if (!hit) {
        hit = victim;
        hit->tick = 0;
        if (!encode_frames_map(&hit->map, dst, dst_pitch, rows, frames, stride, 1, kOutRowBytes, kTileH)) return false;
        hit->base = dst;
        hit->stride = stride;
        hit->frames = frames;
        hit->rows = rows;
    }
    hit->tick = ++p.tick;
    *out = hit->map;
    return true;
}

static void tune_stage(pb_plan& p, cudaStream_t st) {
    if (p.desc.channels != 3) return;
    int h[kProbeInts] = {0};
    if (p.separable && p.tables) {
        // the per-tile footprints are already on the device: histogram them on the host
        const int n_entries = footprint_entries(p);
        int4* host = new (std::nothrow) int4[n_entries];
        if (!host) return;
        if (cudaMemcpyAsync(host, footprint_table(p, p.tables), sizeof(int4) * n_entries, cudaMemcpyDeviceToHost, st) ==
                cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess) {
            for (int e = 0; e < n_entries; ++e) {
                if (host[e].z == 0) continue;
                const int units = stage_units(host[e].w >> 1);
                const int bytes = host[e].z * kBoxRows * 16 * units;
                const bool fits = units <= kMaxStageUnits;
                int bin = (bytes + 1023) >> 10;
                if (!fits || bin > kProbeSizeBins - 1) bin = kProbeSizeBins - 1;
                h[bin] += 1;
                if (fits && units > h[kProbeSizeBins]) h[kProbeSizeBins] = units;
            }
            pick_stage(p, h);
            classify_tiles(p, host, st);
            // single-frame kernel: one buffer holds every rectangle of a tile; size it for 99.5 % of the tiles
            const int nslot = p.src.kind == PB_KIND_DOUBLE ? 2 : 1;
            const int n_tiles = n_entries / nslot;
            int* hist = new (std::nothrow) int[129]();
            if (hist) {
                int counted = 0;
                for (int t = 0; t < n_tiles; ++t) {
                    long long total = 0;
                    for (int s = 0; s < nslot; ++s) {
                        const int4& fp = host[t * nslot + s];
                        if (fp.z == 0) continue;
                        const int units = stage_units(fp.w >> 1);
                        total += units <= kMaxStageUnits ? (long long)fp.z * kBoxRows * 16 * units : (1LL << 40);
                    }
                    if (total == 0) continue;
                    const long long kib = (total + 1023) >> 10;
                    hist[kib > 128 ? 128 : (int)kib] += 1;
                    counted += 1;
                }
                int acc = 0, kib = 128;
                for (int k = 0; k <= 128; ++k) {
                    acc += hist[k];
                    if (acc >= counted - counted / 200) { kib = k; break; }
                }
                if (kib < 4) kib = 4;
                if (kib > 96) kib = 96;
                if (const char* e = std::getenv("PB_SEP1_KIB")) kib = std::atoi(e);  // tuning experiments
                p.sep1_cap = kib * 1024;
                // A third stage buffer (loads issued two tiles ahead instead of one) pays only while four
                // CTAs still fit an SM: T x1 38.2 -> 37.2 us, cfg1 x1 24.9 -> 24.4 us at 13 KiB buffers,
                // slower at 14 KiB (three CTAs) and at 12 KiB (more tiles gather from global memory).
                if (p.src.kind == PB_KIND_CAMERA && counted > 0) {
                    int dev = 0, smem_sm = 0, reserved = 1024;
                    if (cudaGetDevice(&dev) == cudaSuccess &&
                        cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) == cudaSuccess) {
                        (void)cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev);
                        const int budget = smem_sm / PB_SEP1_CAM_CTAS - reserved;
                        int k3 = 0;
                        while (sep1_smem_bytes((k3 + 1) * 1024, false, 3) <= budget) ++k3;
                        int left_out = 0;
                        for (int k = k3 + 1; k <= 128; ++k) left_out += hist[k];
                        if (k3 >= 4 && left_out * 100 <= counted * 3) p.sep1_cap3 = k3 * 1024;
                    }
                    if (const char* e = std::getenv("PB_SEP1_BUFFERS")) {  // tuning experiments
                        if (std::atoi(e) == 2) p.sep1_cap3 = 0;
                        if (std::atoi(e) == 3) p.sep1_cap3 = std::min(p.sep1_cap, 13 * 1024);
                    }
                }
                delete[] hist;
            }
        } else {
            (void)cudaGetLastError();
        }
        delete[] host;
        return;
    }
    int* census = nullptr;
    if (cudaMalloc((void**)&census, sizeof(h)) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    cudaMemsetAsync(census, 0, sizeof(h), st);
    TiledArgs a;
    std::memset(&a, 0, sizeof(a));
    a.out = p.out;
    a.src = p.src;
    a.rot = p.rot;
    a.fast = p.fast;
    a.col_tab = p.tables;
    a.row_tab = p.tables ? p.tables + 2 * (size_t)p.out.W : nullptr;
    a.n_frames = 0;
    a.src_pitch = p.src.W * 3;
    a.stage_bytes = 256;
    a.max_units = kMaxStageUnits;
    a.n_buffers = 1;
    a.n_out = 1;
    a.probe = census;
    a.tiles_x = tiles_x(p);
    a.tiles_y = tiles_y(p);
    a.raster_band = 0;
    if (launch_tiled(a, p.separable && p.tables != nullptr, st) == cudaSuccess &&
        cudaMemcpyAsync(h, census, sizeof(h), cudaMemcpyDeviceToHost, st) == cudaSuccess &&
        cudaStreamSynchronize(st) == cudaSuccess) {
        pick_stage(p, h);
    } else {
        (void)cudaGetLastError();
    }
    cudaFree(census);
}

static cudaError_t fill_tables(const pb_plan& p, double* tables, cudaStream_t st) {
    const int n = p.out.W > p.out.H ? p.out.W : p.out.H;
    pb_tables_kernel<<<(n + 255) / 256, 256, 0, st>>>(p.out, p.src, tables, tables + 2 * (size_t)p.out.W);
    PB_COUNT_LAUNCH();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    TiledArgs a;
    std::memset(&a, 0, sizeof(a));
    a.out = p.out;
    a.src = p.src;
    a.col_tab = tables;
    a.row_tab = tables + 2 * (size_t)p.out.W;
    const int n_entries = footprint_entries(p);
    pb_footprint_kernel<<<(n_entries + 7) / 8, 256, 0, st>>>(a, const_cast<int4*>(footprint_table(p, tables)),
                                                           tiles_x(p), n_entries);
    PB_COUNT_LAUNCH();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int n_tiles = tiles_x(p) * tiles_y(p);
    // launch order of the single-frame kernel: bands of 4 tile rows walked column by column (the
    // resident CTAs then cover a more compact patch of the source than with the 16-row bands of the
    // batched kernel: T x1 37.2 -> 36.8 us)
    static const int sep1_band = env_int("PB_SEP1_RASTER_BAND", 4);
    pb_sep1_table_kernel<<<(n_tiles + 255) / 256, 256, 0, st>>>(footprint_table(p, tables),
                                                              const_cast<int4*>(sep1_table(p, tables)), tiles_x(p),
                                                              tiles_y(p), p.src.kind == PB_KIND_CAMERA ? sep1_band : p.raster_band,
                                                              p.src.kind == PB_KIND_DOUBLE ? 2 : 1);
    PB_COUNT_LAUNCH();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int n_slice = std::max(tiles_x(p) * kTileW, tiles_y(p) * kTileH);
    pb_sep1_slices_kernel<<<(n_slice + 255) / 256, 256, 0, st>>>(tables, tables + 2 * (size_t)p.out.W,
                                                               const_cast<double*>(sep1_col(p, tables)),
                                                               const_cast<double*>(sep1_row(p, tables)), p.out.W, p.out.H,
                                                               tiles_x(p), tiles_y(p), (int)sep1_row_doubles(p));
    PB_COUNT_LAUNCH();
    return cudaGetLastError();
}

// tables: the plan's own, a transient stream-ordered allocation, or null (generic rays)
// [row_begin, row_end): the output rows to produce; dst points at row row_begin (a band of a
// single frame, or the whole image)
static int plan_run(pb_plan& p, const double* tables, const uint8_t* src, int64_t src_frame_stride,
                    uint8_t* dst, int64_t dst_frame_stride, int32_t n_frames, cudaStream_t st, int row_begin = 0,
                    int row_end = -1) {
    std::lock_guard<std::mutex> hold(p.mu);
    if (row_end < 0) row_end = p.out.H;
    const bool whole = row_begin == 0 && row_end == p.out.H;
    const int C = p.desc.channels;
    const long long src_pitch = (long long)p.src.W * C, dst_pitch = (long long)p.out.W * C;
    const bool multi = n_frames > 1;
    const bool tiled_ok = C == 3 && aligned16(src) && aligned16(dst) && src_pitch % 16 == 0 && dst_pitch % 16 == 0 &&
                          (!multi || (src_frame_stride % 16 == 0 && dst_frame_stride % 16 == 0)) &&
                          src_pitch * p.src.H < (1LL << 31);
    // one frame through a non-separable geometry: direct gathers (see remap_direct_kernel)
    static const bool direct_off = std::getenv("PB_DIRECT") && std::atoi(std::getenv("PB_DIRECT")) == 0;  // experiments
    // (a separable geometry takes the tiled kernels when the band starts on a tile row)
    const bool separable_run = p.separable && tables != nullptr && row_begin % kTileH == 0;
    if (n_frames == 1 && !separable_run && !direct_off && C == 3 && p.out.W % 4 == 0 &&
        (reinterpret_cast<uintptr_t>(dst) & 3u) == 0 && src_pitch * p.src.H < (1LL << 31) &&
        (p.out.H + kTileH - 1) / kTileH < 65536) {
        RemapArgs a;
        a.out = p.out;
        a.src = p.src;
        a.rot = p.rot;
        a.fast = p.fast;
        a.src_px = src;
        a.dst_px = dst;
        a.src_frame_stride = src_frame_stride;
        a.dst_frame_stride = dst_frame_stride;
        a.n_frames = 1;
        a.row_begin = row_begin;
        a.row_end = row_end;
        launch_direct(a, st);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return cuda_fail(e, "direct remap launch");
        return PB_OK;
    }
    static const bool tiled_off = std::getenv("PB_TILED") && std::atoi(std::getenv("PB_TILED")) == 0;  // experiments
    if (tiled_ok && !tiled_off && row_begin % kTileH == 0) {
        TiledArgs a;
        std::memset(&a, 0, sizeof(a));
        a.out = p.out;
        a.src = p.src;
        a.rot = p.rot;
        a.fast = p.fast;
        a.col_tab = tables;
        a.row_tab = tables ? tables + 2 * (size_t)p.out.W : nullptr;
        a.tile_fp = tables ? footprint_table(p, tables) : nullptr;
        a.sep1_tab = tables ? sep1_table(p, tables) : nullptr;
        a.sep1_col = tables ? sep1_col(p, tables) : nullptr;
        a.sep1_row = tables ? sep1_row(p, tables) : nullptr;
        a.sep1_cap = p.sep1_cap;
        a.src_px = src;
        a.src_frame_stride = src_frame_stride;
        a.n_frames = n_frames;
        a.src_pitch = (int)src_pitch;
        a.tiles_x = tiles_x(p);
        a.tile_y0 = row_begin / kTileH;
        a.tiles_y = (row_end - row_begin + kTileH - 1) / kTileH;
        a.raster_band = p.raster_band;
        // L2 prefetch (UTMAPF) of frames beyond those in flight: worth +7 % on a single-lens source
        // while tiles kept two frames in flight; with the ring of frame groups it is neutral
        // (8K target) or harmful (double source, -8 %), so it is off  (gpurun_out/run3.log, run12.log)
        a.l2_ahead = 0;
        if (const char* e = std::getenv("PB_L2_AHEAD")) a.l2_ahead = std::atoi(e);  // tuning experiments
        // source rectangles are re-read by neighbouring tiles (keep them), output tiles are written once
        a.load_policy = env_int("PB_LOAD_POLICY", 0);
        a.store_policy = env_int("PB_STORE_POLICY", 2);
        a.lean_min_groups = 1;
        if (const char* e = std::getenv("PB_LEAN_MIN_GROUPS")) a.lean_min_groups = std::atoi(e);  // tuning experiments
#ifdef PB_EXPERIMENTS
        if (const char* e = std::getenv("PB_DEBUG_MODE")) a.debug = std::atoi(e);
#endif
        // stage geometry: one column of 16-row TMA boxes per slot, as wide as the tile needs
        const bool dbl = p.src.kind == PB_KIND_DOUBLE;
        a.stage_bytes = p.stage_bytes;
        a.max_units = p.max_units;
        // a second stage buffer lets the loads of the next (frame, slot) item overlap the current
        // gather; taken when three CTAs per SM still fit
        a.n_out = multi ? 2 : 1;
        a.n_buffers = 1;
        if (multi || dbl) {
            const int mode = (p.separable && tables != nullptr) ? 1 : 0;
            int two;
            if (dbl) two = mode ? tiled_smem_bytes<PB_KIND_DOUBLE, 1>(a.stage_bytes, 2, a.n_out)
                                : tiled_smem_bytes<PB_KIND_DOUBLE, 0>(a.stage_bytes, 2, a.n_out);
            else two = mode ? tiled_smem_bytes<PB_KIND_CAMERA, 1>(a.stage_bytes, 2, a.n_out)
                            : tiled_smem_bytes<PB_KIND_CAMERA, 0>(a.stage_bytes, 2, a.n_out);
            int limit_kib = 75;  // three CTAs per SM
            if (const char* e = std::getenv("PB_TWO_BUF_LIMIT_KIB")) limit_kib = std::atoi(e);  // tuning experiments
            if (two <= limit_kib * 1024) a.n_buffers = 2;
        }
        if (cached_src_maps(p, src, src_pitch, n_frames, src_frame_stride, a.max_units, a.src_maps) &&
            cached_dst_map(p, dst, dst_pitch, row_end - row_begin, n_frames, dst_frame_stride, &a.dst_map)) {
            const bool sep = p.separable && tables != nullptr;
            static const bool sep1_off = std::getenv("PB_SEP1") && std::atoi(std::getenv("PB_SEP1")) == 0;
            cudaError_t e;
            if (sep && whole && n_frames == 1 && !sep1_off && p.out.W / kTileW < 65536 && p.out.H / kTileH < 32768)
            {
                // single-lens source: three stage buffers where the plan found a buffer size that keeps
                // four CTAs per SM (tune_stage), two otherwise
                if (a.src.kind == PB_KIND_CAMERA) {
                    if (p.sep1_cap3 > 0 && tables == p.tables) {
                        a.sep1_cap = p.sep1_cap3;
                        e = launch_sep1_one<PB_KIND_CAMERA, 3>(a, st);
                    } else {
                        e = launch_sep1_one<PB_KIND_CAMERA, 2>(a, st);
                    }
                }
                else if (p.sep1_cls && tables == p.tables && !class_split_off()) {
                    // two grids by tile class, as for batches: the tiles that see both lenses (or the
                    // blend band) keep the two-rectangle buffers, those that see one lens run as a
                    // one-slot kernel with small buffers at four CTAs per SM
                    a.tile_list = p.tile_lists + p.n_one;
                    a.n_list = p.n_rest;
                    a.sep1_tab = p.sep1_cls + p.n_one;
                    pb_plan::SideLane* lane = fork_side(p, st);
                    e = launch_sep1_one<PB_KIND_DOUBLE, 2, 2>(a, lane ? lane->side : st);
                    if (e == cudaSuccess) {
                        a.tile_list = p.tile_lists;
                        a.n_list = p.n_one;
                        a.sep1_tab = p.sep1_cls;
                        a.sep1_cap = env_int("PB_SEP1_ONE_KIB", p.sep1_cap_one >> 10) * 1024;
                        e = launch_sep1_one<PB_KIND_DOUBLE, 2, 1>(a, st);
                    }
                    const cudaError_t ej = join_side(lane, st);  // always: st must not run ahead of the side grid
                    if (e == cudaSuccess) e = ej;
                }
                else
                    e = launch_sep1_one<PB_KIND_DOUBLE, 2>(a, st);
            }
            else if (sep && whole && multi && dbl && p.tile_lists && tables == p.tables && !class_split_off()) {
                // a batch through a double-fisheye source: the tiles that see one lens (small
                // footprints; four CTAs per SM, each with several frames in flight) and the rest
                // (two big rectangles per frame: two CTAs per SM with a stage area twice as large)
                a.n_buffers = 2;
                a.n_out = 2;
                a.tile_list = p.tile_lists + p.n_one;
                a.n_list = p.n_rest;
                a.stage_bytes = env_int("PB_REST_KIB", 50) * 1024;
                pb_plan::SideLane* lane = fork_side(p, st);
                TiledArgs b = a;
                b.tile_list = p.tile_lists;
                b.n_list = p.n_one;
                b.stage_bytes = env_int("PB_ONE_BYTES", 21 * 1024);  // four CTAs per SM
                // the two-lens / blend-band tiles stage the chunks their pixels touch instead of bounding
                // rectangles (pb_chunk.cuh); PB_CHUNK: bit 0 = that class, bit 1 = the one-lens class too
                const int chunk = env_int("PB_CHUNK", 0);
                const int skip = env_int("PB_SKIP_CLASS", 0);  // timing experiments: leave one grid out (wrong output)
                if (skip == 2) {
                    e = cudaSuccess;
                } else if (chunk & 1) {
                    a.stage_bytes = env_int("PB_CHUNK_REST_KIB", 94) * 1024;
                    e = launch_chunk_one<PB_KIND_DOUBLE, 2>(a, lane ? lane->side : st);
                } else if (env_int("PB_CLS2_THREADS", 512) == 512) {
                    // 16 warps per CTA, one quad per thread: twice the warps per SM for the same shared memory
                    // (cfg5 x16: the class alone 0.321 -> 0.301 ms, the step 0.628 -> 0.612 ms)
                    a.stage_bytes = 2 * a.stage_bytes;  // (the ring of frame groups spans what were two stage buffers)
                    e = launch_two_lens(a, lane ? lane->side : st);
                } else {
                    e = launch_tiled_one<PB_KIND_EQUIRECT, PB_KIND_DOUBLE, 1, 2>(a, lane ? lane->side : st);
                }
                if (e == cudaSuccess && skip != 1) {
                    if (chunk & 2) {
                        b.stage_bytes = env_int("PB_CHUNK_ONE_KIB", 38) * 1024;
                        e = launch_chunk_one<PB_KIND_DOUBLE, 1>(b, st);
                    } else {
                        e = launch_tiled_one<PB_KIND_EQUIRECT, PB_KIND_DOUBLE, 1, 1>(b, st);
                    }
                }
                const cudaError_t ej = join_side(lane, st);  // always: st must not run ahead of the side grid
                if (e == cudaSuccess) e = ej;
            }
            else if (sep && whole && multi && !dbl && (env_int("PB_CHUNK", 0) & 4)) {
                a.stage_bytes = env_int("PB_CHUNK_CAM_KIB", 38) * 1024;
                e = launch_chunk_one<PB_KIND_CAMERA, 0>(a, st);
            }
            else
                e = launch_tiled(a, sep, st);
            if (e != cudaSuccess) return cuda_fail(e, "tiled remap launch");
            return PB_OK;
        }
        // no tensor-map encoder in this driver: the generic kernel below needs none
    }
    RemapArgs a;
    a.out = p.out;
    a.src = p.src;
    a.rot = p.rot;
    a.fast = p.fast;
    a.src_px = src;
    a.dst_px = dst;
    a.src_frame_stride = src_frame_stride;
    a.dst_frame_stride = dst_frame_stride;
    a.n_frames = n_frames;
    a.row_begin = row_begin;
    a.row_end = row_end;
    launch_generic(a, st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "generic remap launch");
    return PB_OK;
}

// plan_run for pixels of channels x elem_bytes (2, 4 or 8) bytes, camera / equirect sources: ONE
// launch of remap_wide_kernel for the whole batch (the plan's state is only read: no lock needed)
static int plan_run_wide(const pb_plan& p, int elem_bytes, const void* src, int64_t src_frame_stride, void* dst,
                         int64_t dst_frame_stride, int32_t n_frames, cudaStream_t st, int row_begin = 0,
                         int row_end = -1) {
    if (row_end < 0) row_end = p.out.H;
    const long long tiles_y = (row_end - row_begin + kTileH - 1) / kTileH;
    if (tiles_y >= 65536) return fail(PB_ERR_UNSUPPORTED, "wide remap: more than 65535 x 64 output rows in one call");
    WideArgs a;
    std::memset(&a, 0, sizeof(a));
    a.out = p.out;
    a.src = p.src;
    a.rot = p.rot;
    a.fast = p.fast;
    const bool sep = p.separable && p.tables != nullptr;
    a.col_tab = sep ? p.tables : nullptr;
    a.row_tab = sep ? p.tables + 2 * (size_t)p.out.W : nullptr;
    a.src_px = static_cast<const unsigned char*>(src);
    a.dst_px = static_cast<unsigned char*>(dst);
    a.src_frame_stride = src_frame_stride;
    a.dst_frame_stride = dst_frame_stride;
    a.n_frames = n_frames;
    a.row_begin = row_begin;
    a.row_end = row_end;
    a.px_bytes = p.desc.channels * elem_bytes;
    const int vec = wide_vec(a.px_bytes, src, dst, src_frame_stride, dst_frame_stride, n_frames > 1);
    a.words = a.px_bytes / vec;
    const dim3 grid((p.out.W + kTileW - 1) / kTileW, (unsigned)tiles_y);
    if (sep) {
        launch_wide_v<PB_KIND_EQUIRECT, PB_KIND_CAMERA, true>(a, vec, grid, st);
    } else {
        switch (p.out.kind) {
            case PB_KIND_CAMERA: launch_wide_s<PB_KIND_CAMERA>(a, vec, grid, st); break;
            case PB_KIND_DOUBLE: launch_wide_s<PB_KIND_DOUBLE>(a, vec, grid, st); break;
            default: launch_wide_s<PB_KIND_EQUIRECT>(a, vec, grid, st); break;
        }
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "wide remap launch");
    return PB_OK;
}

// Arguments of the _px entry points that need no device: the element width, then pointers and
// strides against it.  -> PB_OK, or the code with pb_last_error set.
static int check_elem_bytes(int32_t elem_bytes, const char* who) {
    if (elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4 && elem_bytes != 8)
        return fail(PB_ERR_UNSUPPORTED, std::string(who) + ": elem_bytes must be 1, 2, 4 or 8 (got " +
                                            std::to_string(elem_bytes) + ")");
    return PB_OK;
}
static int check_double_source(int src_kind, const char* who) {
    if (src_kind == PB_KIND_DOUBLE)
        return fail(PB_ERR_UNSUPPORTED, std::string(who) +
                                            ": a double-fisheye source blends its two lenses into uint8 "
                                            "(projection.py:459); only elem_bytes == 1 is supported for it");
    return PB_OK;
}
static int check_aligned(const void* p, long long stride, int32_t elem_bytes, const char* who) {
    if ((reinterpret_cast<uintptr_t>(p) % (uintptr_t)elem_bytes) != 0 || stride % elem_bytes != 0)
        return fail(PB_ERR_INVALID_ARGUMENT, std::string(who) + ": pointer or stride not a multiple of elem_bytes");
    return PB_OK;
}

}  // namespace pb

// ------------------------------------------------------------------------------------ C ABI

using namespace pb;

extern "C" {

int pb_version(void) { return PB_ABI_VERSION; }

int64_t pb_kernel_launches(void) { return (int64_t)g_kernel_launches.load(std::memory_order_relaxed); }

const char* pb_last_error(void) { return g_last_error.c_str(); }

int32_t pb_output_width(const pb_image_desc* out) {
    if (!out) return 0;
    return out->kind == PB_KIND_DOUBLE ? 2 * (out->width / 2) : out->width;
}

int pb_remap_u8(const pb_remap_desc* desc, const uint8_t* src, int64_t src_frame_stride, uint8_t* dst,
                int64_t dst_frame_stride, int32_t n_frames, void* stream) {
    if (!src || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_remap_u8: null pointer");
    if (int rc = validate_desc(desc, "pb_remap_u8")) return rc;
    if (n_frames < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_remap_u8: negative n_frames");
    if (n_frames == 0) return PB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    pb_plan p;
    plan_init(p, *desc);
    // no footprint census without a plan: the single-frame tables mark every rectangle of up to
    // kMaxStageUnits units as staged, so a tensor map must exist for every width
    p.max_units = kMaxStageUnits;
    if (cudaError_t e = upload_lens_tables(&desc->out, &p.out, &desc->src, &p.src, &p.luts, st, true))
        return cuda_fail(e, "pb_remap_u8 lens tables");
    double* tables = nullptr;
    if (p.separable) {
        // transient, stream-ordered: nothing outlives the call
        if (cudaMallocAsync((void**)&tables, table_doubles(p) * sizeof(double), st) != cudaSuccess) {
            (void)cudaGetLastError();
            tables = nullptr;  // no memory pool on this device: the generic rays need no tables
        } else if (cudaError_t e = fill_tables(p, tables, st)) {
            cudaFreeAsync(tables, st);
            if (p.luts) cudaFreeAsync(p.luts, st);
            return cuda_fail(e, "pb_remap_u8 tables launch");
        }
    }
    const int rc = plan_run(p, tables, src, src_frame_stride, dst, dst_frame_stride, n_frames, st);
    if (tables) cudaFreeAsync(tables, st);
    if (p.luts) cudaFreeAsync(p.luts, st);
    return rc;
}

// The error bound of the FP32-first tier, K * 2^-24 * shape, holds for every geometry with the K = 16
// of derive_fast32 (calibrated over the lens pairs of the test matrix: the largest ratio seen is
// 6.4).  A plan can do better, and rigorously so: float arithmetic is deterministic, so the
// largest |float - double| / (2^-24 * shape) over THIS plan's own output pixels -- one pass of
// both evaluations at plan creation, ~1 ms for 8K -- bounds the error of exactly the evaluations
// its launches will make.  K_plan = 1.25 * that + 0.25 (typical geometries: 2-5, which cuts the
// pixels that go through the float64 rounds to a quarter); never below 1.5.  A ratio beyond what
// K = 16 covers (none known) raises K instead, and a wild one switches the tier off.
static void calibrate_fast32(pb_plan& p, cudaStream_t st) {
    if (!p.fast.f32.enabled || p.separable) return;  // (separable plans resolve through tables)
    if (std::getenv("PB_FP32_K")) return;            // calibration experiments set K themselves
    if (const char* e = std::getenv("PB_FP32_CALIBRATE")) {
        if (std::atoi(e) == 0) return;
    }
    const Fast32GeomT<double> gd = derive_fast32(p.out, p.src, p.fast);
    RemapArgs a;
    std::memset(&a, 0, sizeof(a));
    a.out = p.out;
    a.src = p.src;
    a.rot = p.rot;
    a.fast = p.fast;
    unsigned* dev = nullptr;
    if (cudaMalloc((void**)&dev, sizeof(unsigned)) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    cudaMemsetAsync(dev, 0, sizeof(unsigned), st);
    switch (a.out.kind) {
        case PB_KIND_CAMERA: launch_ratio_s<PB_KIND_CAMERA>(a, gd, dev, st); break;
        case PB_KIND_DOUBLE: launch_ratio_s<PB_KIND_DOUBLE>(a, gd, dev, st); break;
        default: launch_ratio_s<PB_KIND_EQUIRECT>(a, gd, dev, st); break;
    }
    unsigned bits = 0;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bits, dev, sizeof(bits), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return;  // keep the global bound
    }
    float ratio;
    std::memcpy(&ratio, &bits, sizeof(ratio));
    p.fast32_ratio = ratio;
    if (!(ratio <= 64.0f)) {  // (NaN / inf too)
        p.fast.f32.enabled = 0;
        p.fast32_k = 0.0;
        return;
    }
    p.fast32_k = std::fmax(1.5, 1.25 * (double)ratio + 0.25);
    p.fast.f32.k_eps = (float)(p.fast32_k * 5.9604644775390625e-08);
}

int pb_plan_create(const pb_remap_desc* desc, void* stream, pb_plan** plan_out) {
    if (!plan_out) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_create: null plan pointer");
    *plan_out = nullptr;
    if (int rc = validate_desc(desc, "pb_plan_create")) return rc;
    pb_plan* p = new (std::nothrow) pb_plan;
    if (!p) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_create: out of host memory");
    plan_init(*p, *desc);
    cudaError_t e = cudaGetDevice(&p->device);
    if (e != cudaSuccess) {
        delete p;
        return cuda_fail(e, "pb_plan_create");
    }
    e = upload_lens_tables(&desc->out, &p->out, &desc->src, &p->src, &p->luts, (cudaStream_t)stream, false);
    if (e != cudaSuccess) {
        delete p;
        return cuda_fail(e, "pb_plan_create lens tables");
    }
    p->desc.out.lens_table = p->desc.src.lens_table = nullptr;  // the host tables are the caller's
    if (p->separable) {
        e = cudaMalloc((void**)&p->tables, table_doubles(*p) * sizeof(double));
        if (e == cudaSuccess) e = fill_tables(*p, p->tables, (cudaStream_t)stream);
        if (e != cudaSuccess) {
            if (p->tables) cudaFree(p->tables);
            if (p->luts) cudaFree(p->luts);
            delete p;
            return cuda_fail(e, "pb_plan_create tables");
        }
    }
    calibrate_fast32(*p, (cudaStream_t)stream);
    tune_stage(*p, (cudaStream_t)stream);
    *plan_out = p;
    return PB_OK;
}

int pb_debug_plan_fast32(const pb_plan* plan, double out[2]) {
    if (!plan || !out) return fail(PB_ERR_INVALID_ARGUMENT, "pb_debug_plan_fast32: null pointer");
    out[0] = plan->fast.f32.enabled ? plan->fast32_k : 0.0;
    out[1] = plan->fast32_ratio;
    return PB_OK;
}

int pb_plan_remap_u8(const pb_plan* plan, const uint8_t* src, int64_t src_frame_stride, uint8_t* dst,
                     int64_t dst_frame_stride, int32_t n_frames, void* stream) {
    if (!plan || !src || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_u8: null pointer");
    if (n_frames < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_u8: negative n_frames");
    if (n_frames == 0) return PB_OK;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != plan->device)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_u8: plan belongs to another device");
    return plan_run(*const_cast<pb_plan*>(plan), plan->tables, src, src_frame_stride, dst, dst_frame_stride, n_frames,
                    (cudaStream_t)stream);
}

int pb_plan_remap_rows_u8(const pb_plan* plan, const uint8_t* src, uint8_t* dst_band, int32_t row_begin, int32_t row_end,
                          void* stream) {
    if (!plan || !src || !dst_band) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_u8: null pointer");
    if (row_begin < 0 || row_end > plan->out.H || row_begin > row_end)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_u8: rows outside the output image");
    if (row_begin == row_end) return PB_OK;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != plan->device)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_u8: plan belongs to another device");
    return plan_run(*const_cast<pb_plan*>(plan), plan->tables, src, 0, dst_band, 0, 1, (cudaStream_t)stream, row_begin,
                    row_end);
}

int pb_plan_remap_px(const pb_plan* plan, int32_t elem_bytes, const void* src, int64_t src_frame_stride, void* dst,
                     int64_t dst_frame_stride, int32_t n_frames, void* stream) {
    const char* who = "pb_plan_remap_px";
    if (int rc = check_elem_bytes(elem_bytes, who)) return rc;
    if (!plan || !src || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_px: null pointer");
    if (elem_bytes == 1)
        return pb_plan_remap_u8(plan, static_cast<const uint8_t*>(src), src_frame_stride, static_cast<uint8_t*>(dst),
                                dst_frame_stride, n_frames, stream);
    if (int rc = check_double_source(plan->src.kind, who)) return rc;
    if (int rc = check_aligned(src, src_frame_stride, elem_bytes, who)) return rc;
    if (int rc = check_aligned(dst, dst_frame_stride, elem_bytes, who)) return rc;
    if (n_frames < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_px: negative n_frames");
    if (n_frames == 0) return PB_OK;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != plan->device)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_px: plan belongs to another device");
    return plan_run_wide(*plan, elem_bytes, src, src_frame_stride, dst, dst_frame_stride, n_frames, (cudaStream_t)stream);
}

int pb_plan_remap_rows_px(const pb_plan* plan, int32_t elem_bytes, const void* src, void* dst_band, int32_t row_begin,
                          int32_t row_end, void* stream) {
    const char* who = "pb_plan_remap_rows_px";
    if (int rc = check_elem_bytes(elem_bytes, who)) return rc;
    if (!plan || !src || !dst_band) return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_px: null pointer");
    if (elem_bytes == 1)
        return pb_plan_remap_rows_u8(plan, static_cast<const uint8_t*>(src), static_cast<uint8_t*>(dst_band), row_begin,
                                     row_end, stream);
    if (int rc = check_double_source(plan->src.kind, who)) return rc;
    if (int rc = check_aligned(src, 0, elem_bytes, who)) return rc;
    if (int rc = check_aligned(dst_band, 0, elem_bytes, who)) return rc;
    if (row_begin < 0 || row_end > plan->out.H || row_begin > row_end)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_px: rows outside the output image");
    if (row_begin == row_end) return PB_OK;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != plan->device)
        return fail(PB_ERR_INVALID_ARGUMENT, "pb_plan_remap_rows_px: plan belongs to another device");
    return plan_run_wide(*plan, elem_bytes, src, 0, dst_band, 0, 1, (cudaStream_t)stream, row_begin, row_end);
}

void pb_plan_destroy(pb_plan* plan) {
    if (!plan) return;
    if (plan->tables) cudaFree(plan->tables);
    if (plan->luts) cudaFree(plan->luts);
    if (plan->tile_lists) cudaFree(plan->tile_lists);
    if (plan->sep1_cls) cudaFree(plan->sep1_cls);
    for (int k = 0; k < plan->n_lanes; ++k) {
        cudaStreamDestroy(plan->lanes[k].side);
        cudaEventDestroy(plan->lanes[k].ev_fork);
        cudaEventDestroy(plan->lanes[k].ev_join);
    }
    delete plan;
}

int pb_materialize_map_f64(const pb_remap_desc* desc, double* map, void* stream) {
    if (!desc || !map) return fail(PB_ERR_INVALID_ARGUMENT, "pb_materialize_map_f64: null pointer");
    if (int rc = check_image(desc->out, "out")) return rc;
    if (desc->n_rotations < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_materialize_map_f64: negative n_rotations");
    if (desc->n_rotations > PB_MAX_ROTATIONS)
        return fail(PB_ERR_TOO_MANY_ROTATIONS, "pb_materialize_map_f64: more than PB_MAX_ROTATIONS rotations");
    OutGeom g = derive_out(desc->out);
    Rotations rot;
    rot.n = desc->n_rotations;
    std::memcpy(rot.m, desc->rotations, sizeof(rot.m));
    dim3 block(32, 8);
    dim3 grid((g.W + block.x - 1) / block.x, (g.H + block.y - 1) / block.y);
    cudaStream_t st = (cudaStream_t)stream;
    double* luts = nullptr;
    if (cudaError_t eu = upload_lens_tables(&desc->out, &g, nullptr, nullptr, &luts, st, true))
        return cuda_fail(eu, "pb_materialize_map_f64 lens table");
    switch (g.kind) {
        case PB_KIND_CAMERA: materialize_map_kernel<PB_KIND_CAMERA><<<grid, block, 0, st>>>(g, rot, map); PB_COUNT_LAUNCH(); break;
        case PB_KIND_DOUBLE: materialize_map_kernel<PB_KIND_DOUBLE><<<grid, block, 0, st>>>(g, rot, map); PB_COUNT_LAUNCH(); break;
        default: materialize_map_kernel<PB_KIND_EQUIRECT><<<grid, block, 0, st>>>(g, rot, map); PB_COUNT_LAUNCH(); break;
    }
    cudaError_t e = cudaGetLastError();
    if (luts) cudaFreeAsync(luts, st);
    if (e != cudaSuccess) return cuda_fail(e, "pb_materialize_map_f64 launch");
    return PB_OK;
}

int pb_map_projection_u8(double* map, int32_t map_height, int32_t map_width, uint8_t* dst, void* stream) {
    if (!map || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_map_projection_u8: null pointer");
    if (map_height < 0 || map_width < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_map_projection_u8: negative map size");
    const long long n = (long long)map_height * map_width;
    if (n == 0) return PB_OK;
    if ((n + 255) / 256 > 0x7fffffffLL) return fail(PB_ERR_UNSUPPORTED, "pb_map_projection_u8: map too large");
    cudaStream_t st = (cudaStream_t)stream;
    MapRange* range = nullptr;  // transient, stream-ordered: nothing outlives the call
    cudaError_t e = cudaMallocAsync((void**)&range, sizeof(MapRange), st);
    if (e != cudaSuccess) return cuda_fail(e, "pb_map_projection_u8");
    const MapRange init = {0x7fffffffffffffffLL, (long long)0x8000000000000000ULL, 0, 0};
    e = cudaMemcpyAsync(range, &init, sizeof(init), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        const unsigned blocks = (unsigned)std::min<long long>((n + 255) / 256, 148 * 16);
        map_range_kernel<<<blocks, 256, 0, st>>>(map, n, range);
        PB_COUNT_LAUNCH();
        map_projection_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(map, n, range, dst);
        PB_COUNT_LAUNCH();
        e = cudaGetLastError();
    }
    cudaFreeAsync(range, st);
    if (e != cudaSuccess) return cuda_fail(e, "pb_map_projection_u8 launch");
    return PB_OK;
}

int pb_debug_fast32_stats(const pb_remap_desc* desc, double stats[6], void* stream) {
    if (!stats) return fail(PB_ERR_INVALID_ARGUMENT, "pb_debug_fast32_stats: null pointer");
    if (int rc = validate_desc(desc, "pb_debug_fast32_stats")) return rc;
    pb_plan p;
    plan_init(p, *desc);
    const Fast32GeomT<double> gd = derive_fast32(p.out, p.src, p.fast);
    RemapArgs a;
    std::memset(&a, 0, sizeof(a));
    a.out = p.out;
    a.src = p.src;
    a.rot = p.rot;
    a.fast = p.fast;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* dev = nullptr;
    cudaError_t e = cudaMalloc((void**)&dev, 8 * sizeof(unsigned long long));
    if (e != cudaSuccess) return cuda_fail(e, "pb_debug_fast32_stats");
    cudaMemsetAsync(dev, 0, 8 * sizeof(unsigned long long), st);
    unsigned* maxima = reinterpret_cast<unsigned*>(dev + 4);
    switch (a.out.kind) {
        case PB_KIND_CAMERA: launch_stats_s<PB_KIND_CAMERA>(a, gd, maxima, dev, st); break;
        case PB_KIND_DOUBLE: launch_stats_s<PB_KIND_DOUBLE>(a, gd, maxima, dev, st); break;
        default: launch_stats_s<PB_KIND_EQUIRECT>(a, gd, maxima, dev, st); break;
    }
    unsigned long long host[8];
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(host, dev, sizeof(host), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (e != cudaSuccess) return cuda_fail(e, "pb_debug_fast32_stats");
    float mx[2];
    std::memcpy(mx, host + 4, sizeof(mx));
    stats[0] = mx[0];
    stats[1] = mx[1];
    for (int k = 0; k < 4; ++k) stats[2 + k] = (double)host[k];
    return PB_OK;
}

int pb_rotate_map_f64(const double matrix[9], double* map_in, double* map_out, int64_t n_pixels, void* stream) {
    if (!matrix || !map_in || !map_out) return fail(PB_ERR_INVALID_ARGUMENT, "pb_rotate_map_f64: null pointer");
    if (n_pixels < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_rotate_map_f64: negative n_pixels");
    if (map_in == map_out) return fail(PB_ERR_INVALID_ARGUMENT, "pb_rotate_map_f64: map_in and map_out alias");
    if (n_pixels == 0) return PB_OK;
    Mat3 m;
    std::memcpy(m.m, matrix, sizeof(m.m));
    const int block = 256;
    const long long blocks = (n_pixels + block - 1) / block;
    if (blocks > 0x7fffffffLL) return fail(PB_ERR_UNSUPPORTED, "pb_rotate_map_f64: map too large");
    rotate_map_kernel<<<(unsigned)blocks, block, 0, (cudaStream_t)stream>>>(m, map_in, map_out, n_pixels);
    PB_COUNT_LAUNCH();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "pb_rotate_map_f64 launch");
    return PB_OK;
}

int pb_gather_from_map_u8(const pb_image_desc* src_desc, int32_t channels, double* map, int32_t map_height,
                          int32_t map_width, const uint8_t* src, uint8_t* dst, void* stream) {
    if (!src_desc || !map || !src || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_gather_from_map_u8: null pointer");
    if (int rc = check_image(*src_desc, "src")) return rc;
    // source_lookup packs a source pixel as row << 16 | column
    if (src_desc->height > 32767 || src_desc->width > 65535)
        return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_u8: source larger than 32767 rows x 65535 columns");
    if (channels < 1 || channels > 4) return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_u8: channels must be 1..4");
    if (map_height < 0 || map_width < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_gather_from_map_u8: negative map size");
    const long long n = (long long)map_height * map_width;
    if (n == 0) return PB_OK;
    if ((n + 255) / 256 > 0x7fffffffLL) return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_u8: map too large");
    SrcGeom s = derive_src(*src_desc, channels);
    cudaStream_t st = (cudaStream_t)stream;
    double* luts = nullptr;
    if (cudaError_t eu = upload_lens_tables(nullptr, nullptr, src_desc, &s, &luts, st, true))
        return cuda_fail(eu, "pb_gather_from_map_u8 lens table");
    switch (s.kind) {
        case PB_KIND_CAMERA: launch_gather_c<PB_KIND_CAMERA>(s, map, n, src, dst, st); break;
        case PB_KIND_DOUBLE: launch_gather_c<PB_KIND_DOUBLE>(s, map, n, src, dst, st); break;
        default: launch_gather_c<PB_KIND_EQUIRECT>(s, map, n, src, dst, st); break;
    }
    cudaError_t e = cudaGetLastError();
    if (luts) cudaFreeAsync(luts, st);
    if (e != cudaSuccess) return cuda_fail(e, "pb_gather_from_map_u8 launch");
    return PB_OK;
}

int pb_gather_from_map_px(const pb_image_desc* src_desc, int32_t channels, int32_t elem_bytes, double* map,
                          int32_t map_height, int32_t map_width, const void* src, void* dst, void* stream) {
    const char* who = "pb_gather_from_map_px";
    if (int rc = check_elem_bytes(elem_bytes, who)) return rc;
    if (!src_desc || !map || !src || !dst) return fail(PB_ERR_INVALID_ARGUMENT, "pb_gather_from_map_px: null pointer");
    if (elem_bytes == 1)
        return pb_gather_from_map_u8(src_desc, channels, map, map_height, map_width, static_cast<const uint8_t*>(src),
                                     static_cast<uint8_t*>(dst), stream);
    if (int rc = check_image(*src_desc, "src")) return rc;
    if (int rc = check_double_source(src_desc->kind, who)) return rc;
    if (int rc = check_aligned(src, 0, elem_bytes, who)) return rc;
    if (int rc = check_aligned(dst, 0, elem_bytes, who)) return rc;
    if (src_desc->height > 32767 || src_desc->width > 65535)
        return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_px: source larger than 32767 rows x 65535 columns");
    if (channels < 1 || channels > 4) return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_px: channels must be 1..4");
    if (map_height < 0 || map_width < 0) return fail(PB_ERR_INVALID_ARGUMENT, "pb_gather_from_map_px: negative map size");
    const long long n = (long long)map_height * map_width;
    if (n == 0) return PB_OK;
    if ((n + 255) / 256 > 0x7fffffffLL) return fail(PB_ERR_UNSUPPORTED, "pb_gather_from_map_px: map too large");
    SrcGeom s = derive_src(*src_desc, channels);
    cudaStream_t st = (cudaStream_t)stream;
    double* luts = nullptr;
    if (cudaError_t eu = upload_lens_tables(nullptr, nullptr, src_desc, &s, &luts, st, true))
        return cuda_fail(eu, "pb_gather_from_map_px lens table");
    if (s.kind == PB_KIND_CAMERA) launch_gather_e<PB_KIND_CAMERA>(s, elem_bytes, map, n, src, dst, st);
    else launch_gather_e<PB_KIND_EQUIRECT>(s, elem_bytes, map, n, src, dst, st);
    cudaError_t e = cudaGetLastError();
    if (luts) cudaFreeAsync(luts, st);
    if (e != cudaSuccess) return cuda_fail(e, "pb_gather_from_map_px launch");
    return PB_OK;
}

}  // extern "C"
