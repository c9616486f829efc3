// pb_wide.cuh -- the fused remap for pixels of 2..32 bytes (C = 1..4 channels of 2, 4 or 8-byte
// elements: uint16, float16 / bfloat16, float32, int32, float64 ...), camera and equirect sources.
//
// The reference samples such images by NumPy fancy indexing (projection.py:234-243, 539-546): the
// output pixel is a copy of the source pixel its index picks, in the source's own dtype.  So only
// the byte width of a pixel matters here, and the copy is bit-exact for every dtype: nothing is
// ever converted (NaN payloads, -0.0, infinities and denormals pass through as bytes).
//
// One CTA = one 32 x 64 output tile, 256 threads, in two phases:
//   1. resolve   the source index of each of the tile's 2048 pixels, once per launch, parked in
//                shared memory.  Separable plans (un-rotated equirect output from a camera source)
//                read the plan's tables; every other geometry runs the tier cascade of
//                remap_direct32_kernel: the FP32-first tier on the thread's 8 pixels (4 consecutive
//                pixels in each of two rows), the pixels it leaves undecided deferred to the
//                float64 tiers, one per lane and round.  (With the tier off every pixel is
//                deferred, which is resolve_lookup.)
//   2. gather    per frame of the batch: the 32 lanes of a warp take 32 consecutive pixels of a
//                row, so a warp stores 32 * P contiguous bytes; each pixel moves as NW naturally
//                aligned words of VEC bytes (ld.global.nc), VEC the widest power of two <= 16 that
//                divides P and the alignment of the buffers.  A pixel without a source is zeros.
// One launch covers every frame: the resolve is paid once per tile, not once per frame.
//
// Instantiations: out kind x source kind (+ the separable variant) x VEC; NW (1..4) is a kernel
// argument, its loops fully unrolled and predicated.
#pragma once

#include "pb_device.cuh"
#include "pb_fast32.cuh"
#include "pb_tiled.cuh"

namespace pb {

struct WideArgs {
    OutGeom out;
    SrcGeom src;
    Rotations rot;
    FastGeom fast;
    const double* col_tab;  // separable plans: [W][2] (cos lon_j, sin lon_j)
    const double* row_tab;  // separable plans: [H][4] (lens radius of row i, -, -, -)
    const unsigned char* src_px;
    unsigned char* dst_px;  // points at output row row_begin
    long long src_frame_stride, dst_frame_stride;  // bytes
    int n_frames;
    int row_begin, row_end;  // output rows this launch covers
    int px_bytes;            // P = channels x element bytes
    int words;               // NW = P / VEC
};

template <int VEC> struct WideWord;
template <> struct WideWord<2> { typedef unsigned short T; };
template <> struct WideWord<4> { typedef unsigned T; };
template <> struct WideWord<8> { typedef uint2 T; };
template <> struct WideWord<16> { typedef uint4 T; };

template <typename T> __device__ __forceinline__ T wide_zero();
template <> __device__ __forceinline__ unsigned short wide_zero<unsigned short>() { return 0; }
template <> __device__ __forceinline__ unsigned wide_zero<unsigned>() { return 0u; }
template <> __device__ __forceinline__ uint2 wide_zero<uint2>() { return make_uint2(0u, 0u); }
template <> __device__ __forceinline__ uint4 wide_zero<uint4>() { return make_uint4(0u, 0u, 0u, 0u); }

constexpr int kWideRowsPerWarp = kTileH / 8;  // 8: warp w gathers rows w, w + 8, ..., w + 56 of the tile
constexpr int kWideMaxWords = 4;
// rows whose loads a thread has in flight at once (registers: rows x words of the gather)
#ifndef PB_WIDE_ROWS_IN_FLIGHT
#define PB_WIDE_ROWS_IN_FLIGHT 2
#endif
constexpr int kWideRowsInFlight = PB_WIDE_ROWS_IN_FLIGHT;

// SEP: resolve through the plan's separable tables (OUT_KIND = equirect, SRC_KIND = camera).
// Four CTAs per SM, as remap_direct32_kernel (the float64 tiers fit 64 registers without spills).
#ifndef PB_WIDE_MIN_CTAS
#define PB_WIDE_MIN_CTAS 4
#endif
template <int OUT_KIND, int SRC_KIND, bool SEP, int VEC>
__global__ void __launch_bounds__(256, PB_WIDE_MIN_CTAS) remap_wide_kernel(const __grid_constant__ WideArgs a) {
    static_assert(SRC_KIND != PB_KIND_DOUBLE, "single-slot sources only");
    static_assert(!SEP || (OUT_KIND == PB_KIND_EQUIRECT && SRC_KIND == PB_KIND_CAMERA), "separable: equirect <- camera");
    typedef typename WideWord<VEC>::T Word;
    // source index of tile pixel (r, c) at xys[r][c]; the odd row pitch keeps both the resolve's
    // (4 rows x 8 quads per warp) and the gather's (one row per warp) accesses free of bank conflicts
    __shared__ int xys[kTileH][kTileW + 1];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int row0 = a.row_begin + blockIdx.y * kTileH, col0 = blockIdx.x * kTileW;

    // ---------------------------------------------------------------- 1. resolve
    const int rq = tid >> 3, cq = 4 * (tid & 7);  // quad: pixels (rq + 32 q, cq + k), q < 2, k < 4
    if (SEP) {
#pragma unroll
        for (int q = 0; q < kRowsPerThread; ++q) {
            const int r = rq + q * kRowGroups;
            const int i = min(row0 + r, a.out.H - 1);
            const double dist = __ldg(a.row_tab + 4 * (size_t)i);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int j = min(col0 + cq + k, a.out.W - 1);
                const double2 cs = __ldg(reinterpret_cast<const double2*>(a.col_tab) + j);
                xys[r][cq + k] = camera_xy_from(cs.x, cs.y, dist, a.src.H, a.src.W, a.src.cy, a.src.cx, 0, false);
            }
        }
    } else {
        unsigned pend = 0;  // bit p: pixel p of this thread is left to the float64 tiers
#pragma unroll 1
        for (int q = 0; q < kRowsPerThread; ++q) {
            const int i = row0 + rq + q * kRowGroups;
#pragma unroll 4
            for (int k = 0; k < 4; ++k) {
                const int p = q * 4 + k, j = col0 + cq + k;
                int xy = kNoPixel;
                if (i < a.row_end && j < a.out.W) {
                    Lookup L;
                    if (a.fast.f32.enabled && fast32_lookup<OUT_KIND, SRC_KIND>(a.out, a.fast.f32, a.src, i, j, L)) xy = L.xy0;
                    else pend |= 1u << p;
                }
                xys[rq + q * kRowGroups][cq + k] = xy;
            }
        }
        while (__any_sync(0xffffffffu, pend != 0)) {
            if (pend) {
                const int p = __ffs(pend) - 1;
                pend &= pend - 1;
                const int r = rq + (p >> 2) * kRowGroups, c = cq + (p & 3);
                xys[r][c] = resolve_lookup64<OUT_KIND, SRC_KIND>(a.out, a.fast, a.rot, a.src, row0 + r, col0 + c).xy0;
            }
        }
    }
    __syncthreads();

    // ---------------------------------------------------------------- 2. gather, every frame
    const int j = col0 + lane;
    if (j >= a.out.W) return;
    constexpr int kMaxWords = VEC == 16 ? 2 : kWideMaxWords;  // (P <= 32)
    const int nw = a.words, P = a.px_bytes;
    const long long src_row = (long long)a.src.W * P, dst_row = (long long)a.out.W * P;
    unsigned char* const dst0 = a.dst_px + ((long long)(row0 - a.row_begin + w) * a.out.W + j) * P;
#pragma unroll 1
    for (int f = 0; f < a.n_frames; ++f) {
        const unsigned char* __restrict__ sp = a.src_px + f * a.src_frame_stride;
        unsigned char* __restrict__ dp = dst0 + f * a.dst_frame_stride;
        // groups of kWideRowsInFlight rows: every load of a group is in flight before its first store
#pragma unroll
        for (int g = 0; g < kWideRowsPerWarp; g += kWideRowsInFlight) {
            Word v[kWideRowsInFlight][kMaxWords];
#pragma unroll
            for (int u = 0; u < kWideRowsInFlight; ++u) {
                // (read back per frame: holding the tile's indices in registers across the frame
                // loop costs more registers than the resolve leaves)
                const int r = w + 8 * (g + u);
                const int xy = row0 + r < a.row_end ? xys[r][lane] : kNoPixel;
                const int at = max(xy, 0);
                const Word* s = reinterpret_cast<const Word*>(sp + (at >> 16) * src_row + (at & 0xffff) * P);
#pragma unroll
                for (int n = 0; n < kMaxWords; ++n)
                    v[u][n] = (n < nw && xy >= 0) ? __ldg(s + n) : wide_zero<Word>();
            }
#pragma unroll
            for (int u = 0; u < kWideRowsInFlight; ++u) {
                const int t = g + u;
                if (row0 + w + 8 * t >= a.row_end) break;
                Word* d = reinterpret_cast<Word*>(dp + 8 * t * dst_row);
#pragma unroll
                for (int n = 0; n < kMaxWords; ++n)
                    if (n < nw) d[n] = v[u][n];
            }
        }
    }
}

}  // namespace pb
