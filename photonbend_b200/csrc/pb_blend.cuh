// pb_blend.cuh -- the fused remap of a double-fisheye source of any element type, blended in that
// type (pb_plan_remap_typed / pb_plan_remap_rows_typed): every output element is the reference's
// blend (projection.py:459) with its cast to uint8 replaced by a cast to the source's own type,
// see blend_elem in pb_device.cuh.  (uint8 sources keep their own kernels.)
//
// One CTA = one 32 x 64 output tile, 256 threads, in two phases, as remap_wide_kernel:
//   1. resolve   both lenses' source indices of each of the tile's 2048 pixels, once per launch,
//                parked in shared memory.  Separable plans (un-rotated equirect output) read the
//                plan's tables: the column's (cos, sin) of the longitude and the row's two lens
//                radii; the weights are the row's (row_tab[i][2..3]) and are read per row in the
//                gather.  Every other geometry runs resolve_lookup per pixel (remap_direct_kernel)
//                and parks the two weights beside the indices.
//   2. gather    per frame of the batch: the 32 lanes of a warp take 32 consecutive pixels of a
//                row (a warp stores 32 * P contiguous bytes); each lane loads both lenses' pixels,
//                blends them channel by channel and stores its P bytes.
// One launch covers every frame: the resolve is paid once per tile, not once per frame.
//
// Instantiations: E (element bytes: 1, 2, 4, 8) x (separable, or out kind: 3); the conversions to
// and from float64 switch on the launch's element type at run time.
#pragma once

#include "pb_device.cuh"
#include "pb_fast32.cuh"
#include "pb_tiled.cuh"

namespace pb {

struct BlendArgs {
    OutGeom out;
    SrcGeom src;
    Rotations rot;
    FastGeom fast;
    const double* col_tab;  // separable plans: [W][2] (cos lon_j, sin lon_j)
    const double* row_tab;  // separable plans: [H][4] (left radius, right radius, left weight, right weight)
    const unsigned char* src_px;
    unsigned char* dst_px;  // points at output row row_begin
    long long src_frame_stride, dst_frame_stride;  // bytes
    int n_frames;
    int row_begin, row_end;  // output rows this launch covers
    int channels;            // C = 1..4
    int elem_type;           // PB_ELEM_* (elem_type_bytes(elem_type) == E)
};

template <int E> struct BlendElem;
template <> struct BlendElem<1> { typedef unsigned char T; };
template <> struct BlendElem<2> { typedef unsigned short T; };
template <> struct BlendElem<4> { typedef unsigned T; };
template <> struct BlendElem<8> { typedef unsigned long long T; };

// Four CTAs per SM, as remap_direct_kernel: the per-pixel tiers fit 64 registers without spills
template <int OUT_KIND, bool SEP, int E>
__global__ void __launch_bounds__(256, 4) remap_blend_kernel(const __grid_constant__ BlendArgs a) {
    static_assert(!SEP || OUT_KIND == PB_KIND_EQUIRECT, "separable: equirect output");
    typedef typename BlendElem<E>::T T;
    constexpr int R = E == 8 ? 1 : 2;  // rows whose loads a thread has in flight (more spill at 64 registers)
    // source index of tile pixel (r, c) through lens s at xys[s][r][c]; without separable tables
    // the pixel's two weights at wts[r][c] (48 KB in all: four CTAs per SM)
    __shared__ int xys[2][kTileH][kTileW];
    __shared__ double2 wts[SEP ? 1 : kTileH][kTileW];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int row0 = a.row_begin + blockIdx.y * kTileH, col0 = blockIdx.x * kTileW;

    // ---------------------------------------------------------------- 1. resolve
    const int rq = tid >> 3, cq = 4 * (tid & 7);  // quad: pixels (rq + 32 q, cq + k), q < 2, k < 4
#pragma unroll 1
    for (int q = 0; q < kRowsPerThread; ++q) {
        const int r = rq + q * kRowGroups, i = row0 + r;
        if (SEP) {
            const int ic = min(i, a.out.H - 1);
            const double2 dist = __ldg(reinterpret_cast<const double2*>(a.row_tab) + 2 * (size_t)ic);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int j = min(col0 + cq + k, a.out.W - 1);
                const double2 cs = __ldg(reinterpret_cast<const double2*>(a.col_tab) + j);
                // source_lookup's double-fisheye branch with the radii of the row
                xys[0][r][cq + k] = camera_xy_from(cs.x, cs.y, dist.x, a.src.H, a.src.wl, a.src.cy, a.src.cxl, 0, false);
                xys[1][r][cq + k] = camera_xy_from(cs.x, cs.y, dist.y, a.src.H, a.src.wr, a.src.cy, a.src.cxr, a.src.wl, true);
            }
        } else {
#pragma unroll 1
            for (int k = 0; k < 4; ++k) {
                const int j = col0 + cq + k;
                Lookup L;
                L.xy0 = L.xy1 = kNoPixel;
                L.w0 = L.w1 = 1.0;
                if (i < a.row_end && j < a.out.W) L = resolve_lookup<OUT_KIND, PB_KIND_DOUBLE>(a.out, a.fast, a.rot, a.src, i, j);
                xys[0][r][cq + k] = L.xy0;
                xys[1][r][cq + k] = L.xy1;
                wts[SEP ? 0 : r][cq + k] = make_double2(L.w0, L.w1);
            }
        }
    }
    __syncthreads();

    // ---------------------------------------------------------------- 2. gather, every frame
    const int j = col0 + lane;
    if (j >= a.out.W) return;
    const int C = a.channels, type = a.elem_type, P = C * E;
    const long long src_row = (long long)a.src.W * P, dst_row = (long long)a.out.W * P;
    unsigned char* const dst0 = a.dst_px + ((long long)(row0 - a.row_begin + w) * a.out.W + j) * P;
#pragma unroll 1
    for (int f = 0; f < a.n_frames; ++f) {
        const unsigned char* __restrict__ sp = a.src_px + f * a.src_frame_stride;
        unsigned char* __restrict__ dp = dst0 + f * a.dst_frame_stride;
        // groups of R rows: every load of a group is in flight before its first blend (one row at a
        // time leaves the gather bound by the latency of its loads)
#pragma unroll 1
        for (int g = 0; g < kTileH / 8; g += R) {
            T v0[R][4], v1[R][4];
            double2 wt[R];
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const int r = w + 8 * (g + u);
                const bool in = row0 + r < a.row_end;
                const int xy0 = in ? xys[0][r][lane] : kNoPixel, xy1 = in ? xys[1][r][lane] : kNoPixel;
                if (SEP) wt[u] = __ldg(reinterpret_cast<const double2*>(a.row_tab) + 2 * (size_t)min(row0 + r, a.row_end - 1) + 1);
                else wt[u] = wts[SEP ? 0 : r][lane];
                const T* s0 = reinterpret_cast<const T*>(sp + (max(xy0, 0) >> 16) * src_row + (max(xy0, 0) & 0xffff) * P);
                const T* s1 = reinterpret_cast<const T*>(sp + (max(xy1, 0) >> 16) * src_row + (max(xy1, 0) & 0xffff) * P);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    v0[u][c] = (c < C && xy0 >= 0) ? __ldg(s0 + c) : T(0);
                    v1[u][c] = (c < C && xy1 >= 0) ? __ldg(s1 + c) : T(0);
                }
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const int t = g + u;
                if (row0 + w + 8 * t >= a.row_end) break;
                T* d = reinterpret_cast<T*>(dp + 8 * t * dst_row);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < C) d[c] = (T)blend_elem(v0[u][c], wt[u].x, v1[u][c], wt[u].y, type);
            }
        }
    }
}

}  // namespace pb
