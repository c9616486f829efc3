// pb_tiled.cuh -- the tiled remap kernel (sm_100a), C = 3 uint8 channels.
//
// One CTA = one 32 x 64 tile of the output image (the shape whose source footprint is most
// compact for fisheye <-> equirect mappings, see DESIGN.md), 256 threads, each thread owning two
// "quads" (4 consecutive pixels of a row = 12 output bytes = three 32-bit words).
//
//   1. resolve   every thread resolves the source coordinates of its 8 pixels in float64
//                registers -- either through the generic ray / rotate / lookup functions, or, for
//                an un-rotated equirectangular output, from the separable tables (cos/sin of the
//                column's longitude, lens radius of the row's latitude) that pb_tables_kernel wrote
//                once per geometry.  No coordinate map ever exists in memory.
//   2. footprint the bounding rectangle of the source pixels the tile reads, one per source "slot"
//                (a double-fisheye source has two: left and right lens).  Separable geometry: one
//                warp per slot derives it from the tile's 32 columns x {smallest, largest} lens
//                radius of its rows (the coordinates are monotone in the radius), and learns
//                whether every pixel of the tile is inside the source (then the per-pixel bounds
//                tests are skipped).  Generic rays: warp redux + shared atomics over all pixels.
//   3. stage     for every (frame, slot) item one elected thread pulls the rectangle into shared
//                memory with TMA tensor-map box loads (cp.async.bulk.tensor, 16-row boxes, one
//                mbarrier per stage buffer; the hardware zero-fills what hangs over the image
//                border).  Items rotate through two stage buffers, so the loads of the next item
//                are in flight while the current one is gathered.  Tiles whose footprint does not
//                fit (a pole, the +-pi seam of a panorama) gather straight from global memory.
//   4. gather    threads pick their pixels out of shared memory (two aligned 32-bit loads + a
//                funnel shift per pixel), blend the two slots where the source is a double
//                fisheye, pack 4 pixels into 3 words and write them into the shared output tile.
//   5. store     one TMA tensor-map box store drains the 32 x 64 tile to HBM (clipped by the
//                hardware at the image border), overlapping the next frame's gather.
//
// Steps 1-2 run once per tile, steps 3-5 once per frame: a batch of frames that share a geometry
// pays the float64 index math once.
#pragma once

#include <type_traits>

#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched through the runtime)

#include "pb_device.cuh"
#include "pb_fast32.cuh"
#include "pb_ptx.cuh"

namespace pb {

constexpr int kTileW = 32;
constexpr int kTileH = 64;
constexpr int kTileThreads = 256;
constexpr int kQuadsPerRow = kTileW / 4;                 // 8
constexpr int kRowGroups = kTileThreads / kQuadsPerRow;  // 32
constexpr int kRowsPerThread = kTileH / kRowGroups;      // 2
constexpr int kPxPerThread = 4 * kRowsPerThread;         // 8
constexpr int kOutRowBytes = kTileW * 3;                 // 96
constexpr int kOutTileBytes = kOutRowBytes * kTileH;     // 6144
constexpr int kBoxRows = 16;                             // rows per TMA box of the source map

// A tile stages the bounding rectangle of what it reads with TMA boxes whose width is fixed by
// the tensor map, so there is one map per box width: 16-byte units 5, 7, ... 31 (odd, see
// pick_stage), and a tile takes the narrowest that covers its footprint.
constexpr int kMinStageUnits = 5;
constexpr int kMaxStageUnits = 31;  // u16 tensor map: at most 256 elements per box row
constexpr int kMaxSrcMaps = (kMaxStageUnits - kMinStageUnits) / 2 + 1;  // 14

struct TiledArgs {
    CUtensorMap src_maps[kMaxSrcMaps];  // u16 elements: {pitch/2, H, frames}, box {8 * (5 + 2k), 16, 1}
    CUtensorMap dst_map;  // u8 elements:  {W*3, H, frames},   box {96, 64, 1}
    OutGeom out;
    SrcGeom src;
    Rotations rot;
    FastGeom fast;    // guarded short cut of the per-pixel chain (pb_fast.cuh)
    const double* col_tab;  // separable: [W][2]  (cos lon_j, sin lon_j)
    const double* row_tab;  // separable: [H][4]  camera: (dist, -, -, -); double: (dist_l, dist_r, w_l, w_r)
    const unsigned char* src_px;
    long long src_frame_stride;
    int n_frames;
    int src_pitch;    // bytes per source row
    int stage_bytes;  // capacity of one stage buffer (rows x row pitch of a tile must fit), multiple of 256
    int max_units;    // widest box for which src_maps holds a map, in 16-byte units
    int n_buffers;    // stage buffers: 1, or 2 (loads of the next item overlap the current gather)
    int n_out;        // output tile buffers: 1, or 2 (the store of frame f overlaps frame f+1)
    int* probe;       // non-null: footprint census only (see pb_plan_create), nothing is remapped
    int tiles_x, tiles_y;  // tiles per output row / column (of the row band this launch covers)
    int tile_y0;           // first tile row of the band; the band's first output row is tile_y0 * 64
                           // and dst_map describes the band alone (pb_plan_remap_rows_u8)
    int lean_min_groups;  // tiles that cannot keep this many frames in flight use the (frame, slot) item loop
    int l2_ahead;     // items whose boxes are prefetched into L2 ahead of the shared-memory loads
    int raster_band;  // CTAs walk bands of this many tile rows column by column (0: plain row-major)
    int load_policy, store_policy;  // L2 eviction priority of the staged source / the stored tiles (ptx::policy_of)
#ifdef PB_EXPERIMENTS
    int debug;  // timing experiments (wrong output): 1 = no loads / waits, 2 = no gather, 4 = no stores
#endif
    const int* tile_list;  // non-null: CTA b remaps tile tile_list[b] (a class of tiles, in raster order; n_list CTAs)
    int n_list;
    const int4* tile_fp;  // separable: per (tile, slot) footprint {by0, xb0, nbox, all_valid | need_bytes << 1}
    const int4* tile_box; // separable double-fisheye plan: per (tile, slot, box) extents (pb_boxes.cuh)
    const int4* sep1_tab; // separable: the same per (tile in launch order, slot), pre-decoded (pb_sep1.cuh)
    const double* sep1_col;  // single-frame kernel: per-tile column / row table slices (pb_sep1_slices_kernel)
    const double* sep1_row;
    int sep1_cap;         // single-frame kernel: bytes of source rectangles one stage buffer holds (multiple of 128)
};

// footprint census written by a probe launch: how many (tile, slot) items need a stage buffer of
// k KiB (bin k = (k-1, k] KiB, last bin = more or too wide to stage), then the widest row, in
// 16-byte units, among the items that can be staged
constexpr int kProbeSizeBins = 96;
constexpr int kProbeInts = kProbeSizeBins + 1;

// staged-row pitch of a footprint that is need_bytes wide: an odd number of 16-byte units
__host__ __device__ __forceinline__ int stage_units(int need_bytes) {
    const int u = (need_bytes + 15) >> 4;
    return (u < kMinStageUnits ? kMinStageUnits : u) | 1;
}

// Separable tables for an un-rotated equirect output (a1) feeding a camera (a9) or double (a10)
// source: everything that depends on the column only, or on the row only, evaluated with exactly
// the expressions the per-pixel path uses.
__global__ void __launch_bounds__(256) pb_tables_kernel(const __grid_constant__ OutGeom out,
                                                        const __grid_constant__ SrcGeom src,
                                                        double* __restrict__ col_tab,
                                                        double* __restrict__ row_tab) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < out.W) {
        const double lon = linspace_at(out.x_start, out.x_stop, out.x_step, out.W, t);
        double s, c;
        sincos(lon, &s, &c);
        col_tab[2 * t + 0] = c;
        col_tab[2 * t + 1] = s;
    }
    if (t < out.H) {
        const double lat = linspace_at(out.y_start, out.y_stop, out.y_step, out.H, t);
        double* r = row_tab + 4 * t;
        if (src.kind == PB_KIND_DOUBLE) {
            const double lat_r = __dadd_rn(__dmul_rn(lat, -1.0), kPi);
            r[0] = __dmul_rn(lens_forward(src, lat), src.f);
            r[1] = __dmul_rn(lens_forward(src, lat_r), src.f);
            r[2] = merge_weight(src, lat);
            r[3] = merge_weight(src, lat_r);
        } else {
            r[0] = __dmul_rn(lens_forward(src, lat), src.f);
            r[1] = 0.0;
            r[2] = 1.0;
            r[3] = 1.0;
        }
    }
}

// second word of a gather only where the pixel runs into it: fewer active lanes, fewer bank
// conflicts (8K target x16 0.725 -> 0.744 of the roofline, cfg5 x16 0.503 -> 0.509)
#define PB_LEAN_PICK ptx::lds_pixel_sparse
// ... except for the two-lens / blend-band class of a double-fisheye source, which is bound by its
// own instruction stream at 16 warps per SM, not by the shared-memory pipe (cfg5 by parts,
// profiles/experiments/README.md): there both words are always loaded (3 instructions per gather
// instead of 6).  PB_CLS2_DENSE_PICK=0 to compare.
#ifndef PB_CLS2_DENSE_PICK
#define PB_CLS2_DENSE_PICK 1
#endif
template <bool DENSE>
__device__ __forceinline__ unsigned lean_pick(unsigned word_sa, unsigned offset, unsigned shift) {
    return DENSE ? ptx::lds_pixel(word_sa, offset, shift) : ptx::lds_pixel_sparse(word_sa, offset, shift);
}

constexpr int kMaxGroups = 8;  // frames in flight per tile (lean loop)

struct alignas(16) TileShared {
    uint64_t bar[kMaxGroups];  // one mbarrier per stage buffer (general loop) / frame group (lean loop)
    int min_x[2], max_x[2], min_y[2], max_y[2];
};

__device__ __forceinline__ unsigned pick_px(unsigned stage_sa, int b) {
    // the 3 bytes at byte offset b of the staged rectangle (+ one byte of garbage on top): the
    // aligned word holding the first byte, the next word only when the pixel runs into it, and
    // a funnel shift; SHF takes its shift count modulo 32, so b * 8 does.
    // stage_sa is the (block-uniform) shared-window address of the stage buffer: the loads come
    // out as LDS [R + UR], without a per-pixel address add.
    const unsigned addr = stage_sa + (unsigned)(b & ~3);
    unsigned lo, hi;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.u32 p, %3, 0;\n\t"
        "ld.shared.b32 %0, [%2];\n\t"
        "mov.b32 %1, 0;\n\t"
        "@p ld.shared.b32 %1, [%2+4];\n\t"
        "}"
        : "=r"(lo), "=r"(hi)
        : "r"(addr), "r"(b & 2));
    return __funnelshift_r(lo, hi, b << 3);
}

__device__ __forceinline__ unsigned pick_px_global(const unsigned char* __restrict__ img, int b) {
    return (unsigned)__ldg(img + b) | ((unsigned)__ldg(img + b + 1) << 8) | ((unsigned)__ldg(img + b + 2) << 16);
}

__device__ __forceinline__ unsigned blend_px(unsigned a, double wa, unsigned b, double wb) {
    if (wa == 1.0 && wb == 1.0) return __vadd4(a, b);  // exact: bytes add mod 256 (top byte is garbage anyway)
    unsigned r = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        r |= (unsigned)blend_u8((a >> (8 * c)) & 0xffu, wa, (b >> (8 * c)) & 0xffu, wb) << (8 * c);
    return r;
}

__device__ __forceinline__ unsigned blend_px_weighted(unsigned a, double wa, unsigned b, double wb) {
    unsigned r = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        r |= (unsigned)blend_u8((a >> (8 * c)) & 0xffu, wa, (b >> (8 * c)) & 0xffu, wb) << (8 * c);
    return r;
}

// Fixed-point short cut of the weighted blend (projection.py:459).  The reference truncates
// t = fl(fl(a*wa) + fl(b*wb)), a and b bytes; t is within 1e-13 of the real T = a*wa + b*wb.  With
// the weights rounded to 24 fractional bits, a*ia + b*ib is within 255 units of T * 2^24 (half a
// unit per weight, a, b <= 255) and fits an unsigned word while both weights are >= 0 and their
// sum is <= 1 + 2^-8 (inside the blend band they add up to 1).  So wherever the fixed-point
// fraction is more than 256 units away from an integer its integer part -- the top byte of the
// word -- IS trunc(t); the other ~3e-5 of the channels, and rows whose weights do not qualify (the
// half-degree "safety" strip with its negative weight), take the float64 expression itself.
constexpr int kFixShift = 24;
constexpr unsigned kFixGuard = 257;
__device__ __forceinline__ bool fix_weights(double wa, double wb, unsigned& ia, unsigned& ib) {
    const bool ok = wa >= 0.0 && wb >= 0.0 && wa + wb <= 1.00390625;  // false for NaN
    ia = ok ? (unsigned)__double2int_rn(wa * (double)(1 << kFixShift)) : 0u;
    ib = ok ? (unsigned)__double2int_rn(wb * (double)(1 << kFixShift)) : 0u;
    return ok;
}
__device__ __forceinline__ unsigned blend_px_fix(unsigned a, unsigned ia, double wa, unsigned b, unsigned ib, double wb) {
    unsigned t[3], u[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        t[c] = __byte_perm(a, 0, 0x4440 + c) * ia + __byte_perm(b, 0, 0x4440 + c) * ib;
        // fraction to the top of the word, minus the guard: in range iff guard <= fraction <= 2^24 - guard - 1
        u[c] = t[c] * 256u - (kFixGuard << 8);
    }
    unsigned r = __byte_perm(__byte_perm(t[0], t[1], 0x4473), t[2], 0x4710);  // the three top bytes
    if (max(max(u[0], u[1]), u[2]) >= ((1u << kFixShift) - 2u * kFixGuard) << 8) r = blend_px_weighted(a, wa, b, wb);
    return r;
}

// 4 pixels (low 3 bytes of each word) -> 12 packed bytes
__device__ __forceinline__ void store_quad_sa(unsigned o_sa, const unsigned px[4]) {
    ptx::sts32(o_sa, __byte_perm(px[0], px[1], 0x4210));
    ptx::sts32(o_sa + 4, __byte_perm(px[1], px[2], 0x5421));
    ptx::sts32(o_sa + 8, __byte_perm(px[2], px[3], 0x6542));
}
__device__ __forceinline__ void store_quad(unsigned* o, const unsigned px[4]) {
    o[0] = __byte_perm(px[0], px[1], 0x4210);
    o[1] = __byte_perm(px[1], px[2], 0x5421);
    o[2] = __byte_perm(px[2], px[3], 0x6542);
}

// projection.py:254-259: the float64 coordinates of one camera sample
__device__ __forceinline__ void camera_fxy(double c, double s, double dist, double cy, double cx, double& fx,
                                           double& fy) {
    fx = __dadd_rn(__dmul_rn(c, dist), cx);
    fy = __dadd_rn(-__dmul_rn(s, dist), cy);  // (im * -1) + cy: the negation is exact
}

// trunc(|v|) sits in the low word of |v| + 2^52 rounded toward zero (for |v| < 2^32)
__device__ __forceinline__ int trunc_abs(double v) {
    return __double2loint(__dadd_rz(fabs(v), 4503599627370496.0));
}

// projection.py:223-231: "0 <= trunc(v) < n" is "-1 < v < n" on the reals (NaN fails every compare)
__device__ __forceinline__ bool inside_image(double fx, double fy, int w, int h) {
    return fx > -1.0 && fx < (double)w && fy > -1.0 && fy < (double)h;
}

struct Footprint {
    int mnx, mny, mxx, mxy;
    __device__ __forceinline__ void reset() {
        mnx = mny = 0x7fffffff;
        mxx = mxy = -1;
    }
    __device__ __forceinline__ void add(int x, int y) {
        mnx = min(mnx, x);
        mxx = max(mxx, x);
        mny = min(mny, y);
        mxy = max(mxy, y);
    }
    __device__ __forceinline__ void warp_reduce() {
        mnx = __reduce_min_sync(0xffffffffu, mnx);
        mny = __reduce_min_sync(0xffffffffu, mny);
        mxx = __reduce_max_sync(0xffffffffu, mxx);
        mxy = __reduce_max_sync(0xffffffffu, mxy);
    }
};

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Footprint of one slot of a separable tile, by ONE warp (lane = row pair, then lane = column):
// the source coordinates are monotone in the row's lens radius, so the 32 columns evaluated at
// the smallest and largest radius of the tile's rows bound every pixel of the tile exactly.
__device__ __forceinline__ void separable_footprint(const TiledArgs& a, int slot, int x0, int y0, int lane,
                                                    Footprint& fp, bool& all_valid) {
    const bool dbl = a.src.kind == PB_KIND_DOUBLE;
    const int w = dbl ? (slot ? a.src.wr : a.src.wl) : a.src.W;
    const double cx = dbl ? (slot ? a.src.cxr : a.src.cxl) : a.src.cx;
    // radius range over the 64 rows (NaN radii -- outside a rectilinear lens -- never land anywhere)
    const int ia = min(y0 + lane, a.out.H - 1), ib = min(y0 + lane + 32, a.out.H - 1);
    const double da = __ldg(a.row_tab + 4 * ia + slot), db = __ldg(a.row_tab + 4 * ib + slot);
    const double d_lo = warp_min(fmin(da, db)), d_hi = warp_max(fmax(da, db));
    const int any_nan = __any_sync(0xffffffffu, (da != da) || (db != db));
    // this lane's column at both radii
    const double2 cs = __ldg(reinterpret_cast<const double2*>(a.col_tab) + min(x0 + lane, a.out.W - 1));
    double fxa, fya, fxb, fyb;
    camera_fxy(cs.x, cs.y, d_lo, a.src.cy, cx, fxa, fya);
    camera_fxy(cs.x, cs.y, d_hi, a.src.cy, cx, fxb, fyb);
    const double xlo = fmin(fxa, fxb), xhi = fmax(fxa, fxb), ylo = fmin(fya, fyb), yhi = fmax(fya, fyb);
    const bool hit = xlo < (double)w && xhi > -1.0 && ylo < (double)a.src.H && yhi > -1.0;
    const bool inside = xlo > -1.0 && xhi < (double)w && ylo > -1.0 && yhi < (double)a.src.H;
    fp.reset();
    if (hit) {
        int ixlo = (xlo <= 0.0) ? 0 : __double2int_rz(xlo);
        int ixhi = (xhi >= (double)(w - 1)) ? w - 1 : __double2int_rz(xhi);
        const int iylo = (ylo <= 0.0) ? 0 : __double2int_rz(ylo);
        const int iyhi = (yhi >= (double)(a.src.H - 1)) ? a.src.H - 1 : __double2int_rz(yhi);
        if (slot) {  // right half of a double image, mirrored: column wl + (wr - 1 - px)
            const int t = a.src.W - 1 - ixhi;
            ixhi = a.src.W - 1 - ixlo;
            ixlo = t;
        }
        fp.add(ixlo, iylo);
        fp.add(ixhi, iyhi);
    }
    fp.warp_reduce();
    all_valid = __all_sync(0xffffffffu, inside) && !any_nan;
}

// Footprints of every (tile, slot) of a separable geometry, one warp each; they depend on the
// geometry only, so a plan computes them once (pb_plan_create) and every launch just reads them.
__global__ void __launch_bounds__(256) pb_footprint_kernel(const __grid_constant__ TiledArgs a, int4* __restrict__ tile_fp,
                                                           int tiles_x, int n_entries) {
    const int nslot = (a.src.kind == PB_KIND_DOUBLE) ? 2 : 1;
    const int e = blockIdx.x * 8 + (threadIdx.x >> 5);  // entry = tile * nslot + slot
    if (e >= n_entries) return;
    const int tile = e / nslot, slot = e - tile * nslot;
    const int x0 = (tile % tiles_x) * kTileW, y0 = (tile / tiles_x) * kTileH;
    Footprint fp;
    bool all_valid;
    separable_footprint(a, slot, x0, y0, threadIdx.x & 31, fp, all_valid);
    if ((threadIdx.x & 31) == 0) {
        int4 v = make_int4(0, 0, 0, 0);
        if (fp.mxx >= 0) {
            v.x = fp.mny;
            v.y = (fp.mnx * 3) & ~15;  // TMA: first byte of a box row on a 16-byte boundary
            v.z = (fp.mxy - fp.mny + kBoxRows) / kBoxRows;
            v.w = (all_valid ? 1 : 0) | ((fp.mxx * 3 + 3 - v.y) << 1);
        }
        tile_fp[e] = v;
    }
}

// Slow path of a tile whose footprint cannot be staged (it holds a pole of the source, straddles
// the +-pi seam of a panorama, or is simply too wide): every pixel is resolved again and read
// straight from global memory.  Rare by construction; clarity over speed.
template <int OUT_KIND, int SRC_KIND, int MODE>
__device__ __noinline__ void direct_tile(const TiledArgs& a, const int* xy_scratch, const double2* w_scratch,
                                         unsigned char* out_tile, int x0, int y0) {
    constexpr bool DBL = (SRC_KIND == PB_KIND_DOUBLE);
    const int tid = threadIdx.x;
    for (int f = 0; f < a.n_frames; ++f) {
        const unsigned char* __restrict__ frame = a.src_px + (long long)f * a.src_frame_stride;
        if (f > 0) {
            if (tid == 0) ptx::bulk_wait_read0();
            __syncthreads();
        }
        for (int e = tid; e < kTileW * kTileH; e += (int)blockDim.x) {
            const int r = e / kTileW, c = e - r * kTileW;
            const int i = min(y0 + r, a.out.H - 1), j = min(x0 + c, a.out.W - 1);
            Lookup L;
            if (MODE == 1) {
                // separable tables hold exactly what source_lookup would recompute for this pixel
                const double2 cs = __ldg(reinterpret_cast<const double2*>(a.col_tab) + j);
                const double2 r01 = __ldg(reinterpret_cast<const double2*>(a.row_tab) + 2 * i);
                const double2 r23 = __ldg(reinterpret_cast<const double2*>(a.row_tab) + 2 * i + 1);
                L.xy1 = kNoPixel;
                L.w0 = r23.x;
                L.w1 = r23.y;
                if (DBL) {
                    L.xy0 = camera_xy_from(cs.x, cs.y, r01.x, a.src.H, a.src.wl, a.src.cy, a.src.cxl, 0, false);
                    L.xy1 = camera_xy_from(cs.x, cs.y, r01.y, a.src.H, a.src.wr, a.src.cy, a.src.cxr, a.src.wl, true);
                } else {
                    L.xy0 = camera_xy_from(cs.x, cs.y, r01.x, a.src.H, a.src.W, a.src.cy, a.src.cx, 0, false);
                }
            } else {
                // generic rays were parked in shared memory by the resolve step: pixel e belongs to
                // thread (r % 32) * 8 + c / 4, slot (r / 32) * 4 + c % 4
                const int t = (r & (kRowGroups - 1)) * kQuadsPerRow + (c >> 2);
                const int p = (r / kRowGroups) * 4 + (c & 3);
                L.xy0 = xy_scratch[p * kTileThreads + t];
                L.xy1 = kNoPixel;
                L.w0 = L.w1 = 1.0;
                if (DBL) {
                    L.xy1 = xy_scratch[(kPxPerThread + p) * kTileThreads + t];
                    const double2 w = w_scratch[p * kTileThreads + t];
                    L.w0 = w.x;
                    L.w1 = w.y;
                }
            }
            unsigned v0 = 0, v1 = 0;
            if (L.xy0 >= 0) v0 = pick_px_global(frame, (L.xy0 >> 16) * a.src_pitch + (L.xy0 & 0xffff) * 3);
            if (DBL && L.xy1 >= 0) v1 = pick_px_global(frame, (L.xy1 >> 16) * a.src_pitch + (L.xy1 & 0xffff) * 3);
            const unsigned v = DBL ? blend_px(v0, L.w0, v1, L.w1) : v0;
            unsigned char* o = out_tile + r * kOutRowBytes + c * 3;
            o[0] = (unsigned char)v;
            o[1] = (unsigned char)(v >> 8);
            o[2] = (unsigned char)(v >> 16);
        }
        ptx::fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            ptx::tma_store_3d(&a.dst_map, x0 * 3, y0 - a.tile_y0 * kTileH, f, out_tile);
            ptx::bulk_commit();
        }
    }
    if (tid == 0) ptx::bulk_wait_read0();
}

// MODE: 0 = generic per-pixel rays (any output, any rotations), 1 = separable tables
// CLS (separable double-fisheye source, batches; the plan sorts the tiles into two launches):
//   0 = any tile;
//   1 = tiles that see exactly one lens at unit weights (3 of 4 tiles of a 195-degree pair): one
//       slot, chosen per tile, small footprints, many frames in flight at 4 CTAs per SM;
//   2 = the rest (both lenses, blend band): the code of class 0 at 2 CTAs per SM, i.e. with a
//       stage area large enough to keep several frames of their two big rectangles in flight.
#ifndef PB_ONE_LENS_CTAS
#define PB_ONE_LENS_CTAS 4
#endif
constexpr int tiled_min_ctas(int src_kind, int mode, int cls) {
    return mode != 1 ? 2 : src_kind != PB_KIND_DOUBLE ? 5 : cls == 2 ? 2 : cls == 1 ? PB_ONE_LENS_CTAS : 3;
}
template <int OUT_KIND, int SRC_KIND, int MODE, int CLS = 0>
__global__ void __launch_bounds__(kTileThreads, tiled_min_ctas(SRC_KIND, MODE, CLS))
remap_tiled_kernel(const __grid_constant__ TiledArgs a) {
    constexpr bool DBL = (SRC_KIND == PB_KIND_DOUBLE);
    constexpr bool ONE = DBL && MODE == 1 && CLS == 1;  // one lens per tile, picked at run time
    constexpr int NSLOT = (DBL && !ONE) ? 2 : 1;
    constexpr int S1 = NSLOT - 1;  // index of the second slot (aliases the first when there is none)
    constexpr bool WGT_IN_SMEM = DBL && MODE == 0;  // per-pixel weights live in shared memory

    extern __shared__ __align__(128) unsigned char smem[];
    // [ out tiles: n_out x 6144 ][ stage buffers: n_buffers x (stage_bytes + 128) ][ TileShared ][ scratch ]
    const int buf_bytes = a.stage_bytes + 128;  // + zeroed tail
    const int ztail = buf_bytes - 128;  // where pixels without a source read their black
    unsigned char* out_tiles = smem;
    unsigned char* stages = smem + a.n_out * kOutTileBytes;
    TileShared* sh = reinterpret_cast<TileShared*>(stages + a.n_buffers * buf_bytes);
    int* xy_scratch = reinterpret_cast<int*>(sh + 1);                        // MODE 0: [NSLOT][8][256]
    double2* w_scratch = reinterpret_cast<double2*>(xy_scratch + NSLOT * kPxPerThread * kTileThreads);  // [8][256]

    // thread -> pixels: quad column qc (4 consecutive pixels), rows rg and rg + 32.  A warp then
    // covers 32 columns x 4 consecutive rows, which makes its 12-byte quad stores into the
    // 96-byte-pitch output tile hit 32 distinct banks.
    const int tid = threadIdx.x;
    const int qc = tid & (kQuadsPerRow - 1);
    const int rg = tid >> 3;
    // CTA -> tile.  CTAs are dispatched in blockIdx order, so the tiles that are in flight together
    // should form a compact 2-D patch of the output: their source footprints overlap, and what one
    // CTA pulled into L2 is still there when its neighbours ask for it.  Bands of raster_band tile
    // rows, walked column by column (the last band may be shorter).
    int tile_x, tile_y;
    if (a.tile_list != nullptr) {
        const int t = __ldg(a.tile_list + blockIdx.x);
        tile_y = t / a.tiles_x;
        tile_x = t - tile_y * a.tiles_x;
    } else if (a.raster_band > 0) {
        const int per_band = a.raster_band * a.tiles_x;
        const int band = blockIdx.x / per_band, within = blockIdx.x - band * per_band;
        const int bh = min(a.raster_band, a.tiles_y - band * a.raster_band);
        tile_x = within / bh;
        tile_y = band * a.raster_band + (within - tile_x * bh);
    } else {
        tile_y = blockIdx.x / a.tiles_x;
        tile_x = blockIdx.x - tile_y * a.tiles_x;
    }
    tile_y += a.tile_y0;
    const int x0 = tile_x * kTileW;
    const int y0 = tile_y * kTileH;
    const int ys = y0 - a.tile_y0 * kTileH;  // row of the tile in the destination this launch writes
    const int jx = x0 + 4 * qc;

    if (tid == 0) {
        if (a.probe == nullptr) ptx::prefetch_tensormap(&a.dst_map);
#pragma unroll
        for (int g = 0; g < kMaxGroups; ++g) ptx::mbarrier_init(&sh->bar[g], 1);
        ptx::fence_mbarrier_init();
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            sh->min_x[s] = 0x7fffffff;
            sh->min_y[s] = 0x7fffffff;
            sh->max_x[s] = -1;
            sh->max_y[s] = -1;
        }
    }
    if (tid < a.n_buffers * 8) {
        reinterpret_cast<int4*>(stages + (tid >> 3) * buf_bytes + ztail)[tid & 7] = make_int4(0, 0, 0, 0);
        ptx::fence_async_smem();  // (the lean loop lays the stage area out differently: TMA may write here)
    }

    // ---------------------------------------------------------------- 1. resolve (generic)  2. footprint
    // separable: start the table loads now, they are consumed after the barrier
    double2 cs[4], r01[kRowsPerThread];
    double wrow[kRowsPerThread][2];  // separable double source: blend weights per row
    bool unit_weights = true;        // block-uniform: no pixel of the tile needs a weighted blend
    int4 fpv[NSLOT];
    bool right_lens = false;  // ONE: the tile's lens
    if (MODE == 1) {
        if (ONE) {
            const int4 f0 = __ldg(a.tile_fp + (tile_y * a.tiles_x + tile_x) * 2);
            const int4 f1 = __ldg(a.tile_fp + (tile_y * a.tiles_x + tile_x) * 2 + 1);
            right_lens = f0.z == 0;
            fpv[0] = right_lens ? f1 : f0;
        } else {
#pragma unroll
            for (int s = 0; s < NSLOT; ++s) fpv[s] = __ldg(a.tile_fp + (tile_y * a.tiles_x + tile_x) * NSLOT + s);
        }
        // per-tile slices of the tables in the layout of pb_sep1_slices_kernel: for each of its 4
        // columns a warp reads 128 contiguous bytes (the [W][2] table read at a 64-byte stride cost
        // ~12 L1 wavefronts per LDG.128), rows past the image edge repeat the last row
        {
            const double2* __restrict__ col = reinterpret_cast<const double2*>(a.sep1_col) + tile_x * kTileW;
#pragma unroll
            for (int k = 0; k < 4; ++k) cs[k] = __ldg(col + k * 8 + qc);
#pragma unroll
            for (int q = 0; q < kRowsPerThread; ++q) {
                const int r = tile_y * kTileH + rg + q * kRowGroups;
                if (ONE) {
                    r01[q].x = __ldg(a.sep1_row + 4 * r + (right_lens ? 1 : 0));
                    r01[q].y = 0.0;
                } else if (DBL) {
                    const double2* __restrict__ row = reinterpret_cast<const double2*>(a.sep1_row) + 2 * r;
                    r01[q] = __ldg(row);
                    const double2 r23 = __ldg(row + 1);
                    wrow[q][0] = r23.x;
                    wrow[q][1] = r23.y;
                } else {
                    r01[q].x = __ldg(a.sep1_row + r);
                    r01[q].y = 0.0;
                }
            }
        }
        // barrier init + zeroed tails visible; and: is every blend weight of the tile exactly 1?
        if (DBL && !ONE) {
            bool mine = true;
#pragma unroll
            for (int q = 0; q < kRowsPerThread; ++q) mine = mine && wrow[q][0] == 1.0 && wrow[q][1] == 1.0;
            unit_weights = __syncthreads_and(mine);
#ifdef PB_EXPERIMENTS
            // timing experiments: leave out a class of tiles (16: one lens, 32: both lenses with unit
            // weights, 64: blend band)
            const int cls = (fpv[0].z > 0 && fpv[S1].z > 0) ? (unit_weights ? 32 : 64) : 16;
            if (a.debug & cls) return;
#endif
        } else {
            __syncthreads();
        }
    } else {
        __syncthreads();  // barrier init + zeroed tails + footprint accumulators visible
        // generic rays: heavy float64 code, kept rolled (results parked in shared memory)
        Footprint fp[NSLOT];
        bool mine = true;
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) fp[s].reset();
#pragma unroll 1
        for (int p = 0; p < kPxPerThread; ++p) {
            const int i = min(y0 + rg + (p >> 2) * kRowGroups, a.out.H - 1);
            const int j = min(jx + (p & 3), a.out.W - 1);
            const Lookup L = resolve_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, i, j);
            xy_scratch[p * kTileThreads + tid] = L.xy0;
            if (L.xy0 >= 0) fp[0].add(L.xy0 & 0xffff, L.xy0 >> 16);
            if (DBL) {
                xy_scratch[(kPxPerThread + p) * kTileThreads + tid] = L.xy1;
                w_scratch[p * kTileThreads + tid] = make_double2(L.w0, L.w1);
                mine = mine && L.w0 == 1.0 && L.w1 == 1.0;
                if (L.xy1 >= 0) fp[S1].add(L.xy1 & 0xffff, L.xy1 >> 16);
            }
        }
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) {
            fp[s].warp_reduce();
            if ((tid & 31) == 0 && fp[s].mxx >= 0) {
                atomicMin(&sh->min_x[s], fp[s].mnx);
                atomicMin(&sh->min_y[s], fp[s].mny);
                atomicMax(&sh->max_x[s], fp[s].mxx);
                atomicMax(&sh->max_y[s], fp[s].mxy);
            }
        }
        if (DBL) unit_weights = __syncthreads_and(mine);
        else __syncthreads();
    }

    // rectangle of slot s: rows [by0, by0 + 16*nbox), bytes [xb0, xb0 + pitch) of each row
    int by0[NSLOT], xb0[NSLOT], nbox[NSLOT], pitch[NSLOT];
    bool all_valid[NSLOT];
    bool staged = true;  // every rectangle fits a stage buffer (what the (frame, slot) item loop needs)
    bool wide = false;   // some rectangle is wider than any tensor map: cannot be staged at all
#pragma unroll
    for (int s = 0; s < NSLOT; ++s) {
        int need_bytes = 0;
        by0[s] = xb0[s] = nbox[s] = 0;
        pitch[s] = 16 * kMinStageUnits;
        all_valid[s] = false;
        if (MODE == 1) {
            by0[s] = fpv[s].x;
            xb0[s] = fpv[s].y;
            nbox[s] = fpv[s].z;
            all_valid[s] = fpv[s].w & 1;
            need_bytes = fpv[s].w >> 1;
        } else {
            const int hi_x = sh->max_x[s];
            if (hi_x >= 0) {
                by0[s] = sh->min_y[s];
                // TMA needs the first byte of a box row on a 16-byte boundary (measured: any other
                // start faults with "illegal instruction", profiles/microbench/tma_probe.cu)
                xb0[s] = (sh->min_x[s] * 3) & ~15;
                nbox[s] = (sh->max_y[s] - by0[s] + kBoxRows) / kBoxRows;
                need_bytes = hi_x * 3 + 3 - xb0[s];
            }
        }
        if (nbox[s] == 0) continue;
        // the narrowest box that covers the footprint
        // (the funnel-shift gather may read a few bytes past a pixel: the next row, or the tail)
        const int units = stage_units(need_bytes);
        pitch[s] = 16 * units;
        const int bytes = nbox[s] * kBoxRows * pitch[s];
        if (units > a.max_units) wide = true;
        if (units > a.max_units || bytes > a.stage_bytes) staged = false;
        if (a.probe != nullptr && tid == 0) {
            const bool fits = units <= kMaxStageUnits;
            atomicAdd(a.probe + (fits ? min((bytes + 1023) >> 10, kProbeSizeBins - 1) : kProbeSizeBins - 1), 1);
            if (fits) atomicMax(a.probe + kProbeSizeBins, units);
        }
    }
    if (a.probe != nullptr) return;

    // ---------------------------------------------------------------- 3. stage (issued first: the loads fly while the offsets are resolved)
    // items = (frame, active slot) pairs, in order; item t uses stage buffer t % n_buffers
    const int first = (nbox[0] > 0) ? 0 : S1;
    const int n_act = (nbox[0] > 0) + ((NSLOT == 2 && nbox[S1] > 0) ? 1 : 0);
    const int n_items = a.n_frames * n_act;
    auto issue_item = [&](int t) {  // one thread
        const int b = (a.n_buffers == 2) ? (t & 1) : 0;
        const int s = (n_act == 2) ? (t & 1) : first;
        const int f = (n_act == 2) ? (t >> 1) : t;
        ptx::mbarrier_arrive_expect_tx(&sh->bar[b], (unsigned)(nbox[s] * kBoxRows * pitch[s]));
        const uint64_t keep = ptx::policy_evict_last();
        const CUtensorMap* map = &a.src_maps[(pitch[s] >> 5) - (kMinStageUnits >> 1)];
        for (int k = 0; k < nbox[s]; ++k)
            ptx::tma_load_3d_hint(stages + b * buf_bytes + k * kBoxRows * pitch[s], map, xb0[s] >> 1,
                                  by0[s] + k * kBoxRows, f, &sh->bar[b], keep);
    };
    // DRAM latency is hidden one level up: the boxes of the items l2_ahead further on are pulled
    // into L2 by prefetches (they need no shared memory), so the loads proper mostly hit L2
    auto prefetch_item = [&](int t) {  // one thread
        const int s = (n_act == 2) ? (t & 1) : first;
        const int f = (n_act == 2) ? (t >> 1) : t;
        const CUtensorMap* map = &a.src_maps[(pitch[s] >> 5) - (kMinStageUnits >> 1)];
        for (int k = 0; k < nbox[s]; ++k) ptx::tma_prefetch_l2_3d(map, xb0[s] >> 1, by0[s] + k * kBoxRows, f);
    };
#ifdef PB_EXPERIMENTS
    const bool dbg_noload = a.debug & 1, dbg_nogather = a.debug & 2, dbg_nostore = a.debug & 4;
#else
    constexpr bool dbg_noload = false, dbg_nogather = false, dbg_nostore = false;
#endif
    // The common case -- no weighted blend anywhere in the tile -- runs the lean frame loop further
    // down.  It treats the stage area as a ring of frame groups: [128 zero bytes][slot 0 rectangle]
    // [slot 1 rectangle], as many as fit, each with its own mbarrier, so that a tile with a small
    // footprint keeps more frames in flight than one with a large footprint.
    const int rect0 = nbox[0] * kBoxRows * pitch[0];
    const int rect1 = (NSLOT == 2) ? nbox[S1] * kBoxRows * pitch[S1] : 0;
    const int group_bytes = 128 + rect0 + rect1;
    int n_groups = min(min(kMaxGroups, a.n_frames), (a.n_buffers * buf_bytes) / group_bytes);
#ifdef PB_EXPERIMENTS
    if (a.debug >> 8) n_groups = min(n_groups, a.debug >> 8);
#endif
    // (separable double source: tiles of the blend band run it too, with the per-row weighted blend)
    // (the lean loop only needs one frame's rectangles to fit the whole stage area)
    const bool lean = (unit_weights || (MODE == 1 && DBL && !ONE)) && n_act >= 1 && n_groups >= a.lean_min_groups &&
                      !wide && (a.n_out == 2 || a.n_frames == 1);  // (the timing experiments apply to either loop)
    if (!staged && !lean) {  // block-uniform
        direct_tile<OUT_KIND, SRC_KIND, MODE>(a, xy_scratch, w_scratch, out_tiles, x0, y0);
        return;
    }
    auto issue_group = [&](int f, int g) {  // one thread: every rectangle of frame f into group g
        unsigned char* base = stages + g * group_bytes + 128;
        ptx::mbarrier_arrive_expect_tx(&sh->bar[g], (unsigned)(rect0 + rect1));
        const uint64_t keep = ptx::policy_of(a.load_policy);
        if (nbox[0] > 0) {
            const CUtensorMap* map = &a.src_maps[(pitch[0] >> 5) - (kMinStageUnits >> 1)];
            for (int k = 0; k < nbox[0]; ++k)
                ptx::tma_load_3d_hint(base + k * kBoxRows * pitch[0], map, xb0[0] >> 1, by0[0] + k * kBoxRows, f, &sh->bar[g],
                                      keep);
        }
        if (NSLOT == 2 && nbox[S1] > 0) {
            const CUtensorMap* map = &a.src_maps[(pitch[S1] >> 5) - (kMinStageUnits >> 1)];
            for (int k = 0; k < nbox[S1]; ++k)
                ptx::tma_load_3d_hint(base + rect0 + k * kBoxRows * pitch[S1], map, xb0[S1] >> 1, by0[S1] + k * kBoxRows, f,
                                      &sh->bar[g], keep);
        }
    };
    auto prefetch_group = [&](int f) {  // one thread: frame f into L2
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) {
            const CUtensorMap* map = &a.src_maps[(pitch[s] >> 5) - (kMinStageUnits >> 1)];
            for (int k = 0; k < nbox[s]; ++k) ptx::tma_prefetch_l2_3d(map, xb0[s] >> 1, by0[s] + k * kBoxRows, f);
        }
    };
    if (lean) {
        if (tid < n_groups * 8) reinterpret_cast<int4*>(stages + (tid >> 3) * group_bytes)[tid & 7] = make_int4(0, 0, 0, 0);
        if (tid == 0 && !dbg_noload) {
            for (int f = 0; f < n_groups; ++f) issue_group(f, f);
            for (int f = n_groups; f < min(n_groups + a.l2_ahead, a.n_frames); ++f) prefetch_group(f);
        }
    } else if (tid == 0 && !dbg_noload) {
        for (int t = 0; t < min(a.n_buffers, n_items); ++t) issue_item(t);
        for (int t = a.n_buffers; t < min(a.n_buffers + a.l2_ahead, n_items); ++t) prefetch_item(t);
    }

    // ---------------------------------------------------------------- 1. resolve (separable) -> byte offsets
    // loc = byte offset of the pixel inside the staged rectangle of its slot (ztail: no source)
    int loc[NSLOT][kPxPerThread];
    // "no source pixel": the zeroed tail of the stage buffer in the item loop; the lean loop may
    // stage rectangles larger than a stage buffer, where ztail is a real offset, so it marks with -1
    const int no_px = lean ? -1 : ztail;
    if (MODE == 1) {
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) {
            const bool right = ONE ? right_lens : (s != 0);  // right half of a double image: mirrored columns
            const int w = DBL ? (right ? a.src.wr : a.src.wl) : a.src.W;
            const double cx = DBL ? (right ? a.src.cxr : a.src.cxl) : a.src.cx;
            const int origin = by0[s] * pitch[s] + xb0[s];
            if (nbox[s] == 0) {  // nothing of this slot is visible from the tile
#pragma unroll
                for (int p = 0; p < kPxPerThread; ++p) loc[s][p] = no_px;
            } else if (all_valid[s]) {  // every pixel lands inside the source: no bounds tests
#pragma unroll
                for (int q = 0; q < kRowsPerThread; ++q)
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        double fx, fy;
                        camera_fxy(cs[k].x, cs[k].y, s ? r01[q].y : r01[q].x, a.src.cy, cx, fx, fy);
                        int px = trunc_abs(fx);
                        if (right) px = a.src.W - 1 - px;
                        loc[s][q * 4 + k] = trunc_abs(fy) * pitch[s] + (px * 3 - origin);
                    }
            } else {
#pragma unroll
                for (int q = 0; q < kRowsPerThread; ++q)
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        double fx, fy;
                        camera_fxy(cs[k].x, cs[k].y, s ? r01[q].y : r01[q].x, a.src.cy, cx, fx, fy);
                        int px = trunc_abs(fx);
                        if (right) px = a.src.W - 1 - px;
                        const int off = trunc_abs(fy) * pitch[s] + (px * 3 - origin);
                        loc[s][q * 4 + k] = inside_image(fx, fy, w, a.src.H) ? off : no_px;
                    }
            }
        }
    } else {
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) {
            const int origin = by0[s] * pitch[s] + xb0[s];
#pragma unroll
            for (int p = 0; p < kPxPerThread; ++p) {
                const int v = xy_scratch[(s * kPxPerThread + p) * kTileThreads + tid];
                loc[s][p] = (v >= 0) ? (v >> 16) * pitch[s] + (v & 0xffff) * 3 - origin : no_px;
            }
        }
    }

    // ---------------------------------------------------------------- 4. gather  5. store (lean loop)
    // Everything is hoisted: per pixel and slot two LDS and one funnel shift, per frame one block
    // barrier; thread 0 refills the group and stores the tile right after it.
    const unsigned stages_sa = ptx::smem_addr(stages);
    if (lean) {
        const uint64_t drop = ptx::policy_of(a.store_policy);
        const unsigned out_sa = ptx::smem_addr(out_tiles) + rg * kOutRowBytes + qc * 12;
        const unsigned out_flip = (a.n_out == 2) ? kOutTileBytes : 0;
        const unsigned bar_sa = ptx::smem_addr(&sh->bar[0]);
        // loc -> address inside a group (pixels without a source read the group's zero bytes)
        unsigned adr[NSLOT][kPxPerThread], shf[NSLOT][kPxPerThread];
#pragma unroll
        for (int s = 0; s < NSLOT; ++s)
#pragma unroll
            for (int p = 0; p < kPxPerThread; ++p) {
                const int l = loc[s][p];
                const int rel = (l == no_px) ? 0 : l + 128 + (s ? rect0 : 0);
                adr[s][p] = stages_sa + (unsigned)(rel & ~3);
                shf[s][p] = (unsigned)rel << 3;
            }
        // blend band: per row of this thread, 0 = unit weights (exact byte add), 1 = fixed-point
        // short cut with float64 fall-back, 2 = float64 only
        unsigned wfix[kRowsPerThread][2];
        int wmode[kRowsPerThread];
#pragma unroll
        for (int q = 0; q < kRowsPerThread; ++q) {
            wfix[q][0] = wfix[q][1] = 0;
            wmode[q] = 0;
            if (MODE == 1 && DBL && !ONE && !unit_weights && !(wrow[q][0] == 1.0 && wrow[q][1] == 1.0))
                wmode[q] = fix_weights(wrow[q][0], wrow[q][1], wfix[q][0], wfix[q][1]) ? 1 : 2;
        }
        __syncthreads();  // the groups' zero bytes are in place
        constexpr bool DENSE = (CLS == 2) && (PB_CLS2_DENSE_PICK != 0);
        auto frame_loop = [&](auto ACT, auto WGT) {
            constexpr int act = decltype(ACT)::value;  // 1: slot 0 only, 2: slot 1 only, 3: both
            constexpr bool wgt = decltype(WGT)::value;  // some row of the tile has a weighted blend
            int g = 0;
            unsigned parity = 0;
            for (int f = 0; f < a.n_frames; ++f) {
                const unsigned goff = (unsigned)(g * group_bytes);
                if (!dbg_noload) ptx::mbarrier_wait_sa(bar_sa + 8 * g, parity);
                unsigned v[kPxPerThread];
                if (dbg_nogather) {
#pragma unroll
                    for (int p = 0; p < kPxPerThread; ++p) v[p] = adr[0][p] + f;
                } else if (wgt) {
                    unsigned w[kPxPerThread];
#pragma unroll
                    for (int p = 0; p < kPxPerThread; ++p) {
                        v[p] = (act & 1) ? lean_pick<DENSE>(adr[0][p], goff, shf[0][p]) : 0u;
                        w[p] = (act & 2) ? lean_pick<DENSE>(adr[S1][p], goff, shf[S1][p]) : 0u;
                    }
#pragma unroll
                    for (int q = 0; q < kRowsPerThread; ++q) {
                        if (wmode[q] == 0) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) v[q * 4 + k] = __vadd4(v[q * 4 + k], w[q * 4 + k]);
                        } else if (wmode[q] == 1) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                v[q * 4 + k] = blend_px_fix(v[q * 4 + k], wfix[q][0], wrow[q][0], w[q * 4 + k], wfix[q][1],
                                                            wrow[q][1]);
                        } else {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                v[q * 4 + k] = blend_px_weighted(v[q * 4 + k], wrow[q][0], w[q * 4 + k], wrow[q][1]);
                        }
                    }
                } else {
                    if (act & 1) {
#pragma unroll
                        for (int p = 0; p < kPxPerThread; ++p) v[p] = lean_pick<DENSE>(adr[0][p], goff, shf[0][p]);
                    }
                    if (act & 2) {
#pragma unroll
                        for (int p = 0; p < kPxPerThread; ++p) {
                            const unsigned w = lean_pick<DENSE>(adr[S1][p], goff, shf[S1][p]);
                            v[p] = (act & 1) ? __vadd4(v[p], w) : w;
                        }
                    }
                }
                const unsigned o = out_sa + (f & 1) * out_flip;
#pragma unroll
                for (int q = 0; q < kRowsPerThread; ++q) store_quad_sa(o + q * kRowGroups * kOutRowBytes, v + q * 4);
                ptx::fence_async_smem();
                if (tid == 0) ptx::bulk_wait_read0();  // stores up to frame f - 1 have left their tiles
                __syncthreads();
                if (tid == 0) {
                    if (f + n_groups < a.n_frames && !dbg_noload) issue_group(f + n_groups, g);
                    if (!dbg_nostore) ptx::tma_store_3d_hint(&a.dst_map, x0 * 3, ys, f, out_tiles + (f & 1) * out_flip, drop);
                    ptx::bulk_commit();
                    if (a.l2_ahead > 0 && f + n_groups + a.l2_ahead < a.n_frames) prefetch_group(f + n_groups + a.l2_ahead);
                }
                if (++g == n_groups) {
                    g = 0;
                    parity ^= 1u;
                }
            }
        };
        if (MODE == 1 && DBL && !ONE && !unit_weights) {
            if (n_act == 2) frame_loop(std::integral_constant<int, 3>{}, std::true_type{});
            else if (first == 0) frame_loop(std::integral_constant<int, 1>{}, std::true_type{});
            else frame_loop(std::integral_constant<int, 2>{}, std::true_type{});
        } else if (n_act == 2) frame_loop(std::integral_constant<int, 3>{}, std::false_type{});
        else if (first == 0) frame_loop(std::integral_constant<int, 1>{}, std::false_type{});
        else frame_loop(std::integral_constant<int, 2>{}, std::false_type{});
        if (tid == 0) ptx::bulk_wait_read0();
        return;
    }

    // ---------------------------------------------------------------- 4. gather  5. store (general loop)
    int t = 0;
    for (int f = 0; f < a.n_frames; ++f) {
        // v = the frame's pixels: slot 0 as gathered, then (double source) blended with slot 1 in place
        unsigned v[kPxPerThread];
#pragma unroll
        for (int s = 0; s < NSLOT; ++s) {
            if (nbox[s] == 0) {  // block-uniform: this slot contributes black
#pragma unroll
                for (int p = 0; p < kPxPerThread; ++p) {
                    if (s == 0) v[p] = 0;
                    else if (WGT_IN_SMEM) {
                        const double2 w = w_scratch[p * kTileThreads + tid];
                        v[p] = blend_px(v[p], w.x, 0u, w.y);
                    } else v[p] = blend_px(v[p], wrow[p >> 2][0], 0u, wrow[p >> 2][1]);
                }
                continue;
            }
            const int b = (a.n_buffers == 2) ? (t & 1) : 0;
            if (!dbg_noload) ptx::mbarrier_wait(&sh->bar[b], (unsigned)((a.n_buffers == 2 ? (t >> 1) : t) & 1));
            const unsigned stage_sa = stages_sa + b * buf_bytes;
            // all loads of the item first (they are independent), then the blends
            unsigned g[kPxPerThread];
#pragma unroll
            for (int p = 0; p < kPxPerThread; ++p) g[p] = dbg_nogather ? 0u : pick_px(stage_sa, loc[s][p]);
            if (s == 0) {
#pragma unroll
                for (int p = 0; p < kPxPerThread; ++p) v[p] = g[p];
            } else if (WGT_IN_SMEM) {
#pragma unroll
                for (int p = 0; p < kPxPerThread; ++p) {
                    const double2 w = w_scratch[p * kTileThreads + tid];
                    v[p] = blend_px(v[p], w.x, g[p], w.y);
                }
            } else {
#pragma unroll
                for (int q = 0; q < kRowsPerThread; ++q) {
                    if (wrow[q][0] == 1.0 && wrow[q][1] == 1.0) {  // outside the blend band: exact byte add
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[q * 4 + k] = __vadd4(v[q * 4 + k], g[q * 4 + k]);
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            v[q * 4 + k] = blend_px_weighted(v[q * 4 + k], wrow[q][0], g[q * 4 + k], wrow[q][1]);
                    }
                }
            }
            // every thread is done with this stage buffer (and, once per frame, the store that last
            // read this frame's output tile is done with it)
            if (tid == 0 && s == S1 && f >= a.n_out) {
                if (a.n_out == 2) ptx::bulk_wait_read1();
                else ptx::bulk_wait_read0();
            }
            __syncthreads();
            if (tid == 0 && !dbg_noload) {
                if (t + a.n_buffers < n_items) issue_item(t + a.n_buffers);
                if (a.l2_ahead > 0 && t + a.n_buffers + a.l2_ahead < n_items) prefetch_item(t + a.n_buffers + a.l2_ahead);
            }
            ++t;
        }
        if (n_act == 0 || (NSLOT == 2 && nbox[S1] == 0)) {
            // the wait above was skipped: still order the reuse of the output tile
            if (f >= a.n_out) {
                if (tid == 0) {
                    if (a.n_out == 2) ptx::bulk_wait_read1();
                    else ptx::bulk_wait_read0();
                }
                __syncthreads();
            }
        }

        unsigned char* out_tile = out_tiles + ((a.n_out == 2) ? (f & 1) : 0) * kOutTileBytes;
#pragma unroll
        for (int q = 0; q < kRowsPerThread; ++q)
            store_quad(reinterpret_cast<unsigned*>(out_tile + (rg + q * kRowGroups) * kOutRowBytes + qc * 12), v + q * 4);
        ptx::fence_async_smem();
        __syncthreads();
        if (tid == 0 && !dbg_nostore) {
            ptx::tma_store_3d_hint(&a.dst_map, x0 * 3, ys, f, out_tile, ptx::policy_evict_first());
            ptx::bulk_commit();
        }
    }
    if (tid == 0) ptx::bulk_wait_read0();
}

template <int SRC_KIND, int MODE>
inline int tiled_smem_bytes(int stage_bytes, int n_buffers, int n_out) {
    const int nslot = (SRC_KIND == PB_KIND_DOUBLE) ? 2 : 1;
    int bytes = n_out * kOutTileBytes + n_buffers * (stage_bytes + 128) + (int)sizeof(TileShared);
    if (MODE == 0) {
        bytes += nslot * kPxPerThread * kTileThreads * (int)sizeof(int);
        if (SRC_KIND == PB_KIND_DOUBLE) bytes += kPxPerThread * kTileThreads * (int)sizeof(double2);
    }
    return bytes + 128;
}

}  // namespace pb
