// pb_frames.cuh -- a batch whose every frame has a rotation of its own (pb_plan_remap_frames_px):
// frame k is remapped as if the plan's rotations R_1 .. R_n were followed by M_k, i.e. the
// reference's protocol with one more rotate_coordinate_map call per frame:
//
//     out_k = src.process_coordinate_map(Rotation_k.rotate_coordinate_map(R_n(... R_1(dst.get_coordinate_map()))))
//
// (stabilised or levelled 360-degree video, a virtual camera moving through a panorama).
//
// One CTA = one 32 x 64 output tile of ONE frame, 256 threads; the grid's z axis runs over the
// frames of the launch.  Each CTA first builds its frame's FastGeom and Rotations in shared memory:
// the constants every frame shares (derived on the host for n + 1 rotations) with the three things
// that differ per frame patched in -- the composed matrix M_k R_n ... R_1 (and its float copy), the
// tiers' enabled flags (a non-orthonormal or non-finite M_k takes the exact chain), and M_k as the
// exact chain's last rotation.  Then the tier cascade of the one-rotation kernels:
//   camera / equirect source   the FP32-first tier on the thread's 8 pixels, the pixels it leaves
//                              undecided deferred to the float64 tiers one per lane and round
//                              (remap_direct32_kernel / remap_wide_kernel), indices parked in shared
//                              memory; then the gather of remap_wide_kernel: a warp moves 32
//                              consecutive pixels of a row as naturally aligned words of VEC bytes.
//   double-fisheye source      resolve_lookup in place and the blend of the two lenses
//                              (remap_direct_kernel), channel by channel: blend_u8, or for a source
//                              that keeps its type the typed blend (blend_px_typed).
// The per-pixel functions are the ones every other kernel calls, so frame k is byte-identical to
// the plan path for a descriptor with M_k appended to its rotations.
//
// The per-frame data travel in the __grid_constant__ kernel parameter (nothing is allocated or
// copied, so a call can be captured into a CUDA graph): kFramesPerLaunch = 128 frames of 192 bytes
// fit the 32 KB parameter space of sm_70+ with the shared constants; a larger batch is launched in
// chunks of 128 frames.
//
// Instantiations: out kind x source kind (9); the gather's word width is a runtime switch.
#pragma once

#include "pb_device.cuh"
#include "pb_fast32.cuh"
#include "pb_tiled.cuh"
#include "pb_wide.cuh"

namespace pb {

// What differs from one frame of the batch to the next.
struct FrameRotation {
    double rot[9];    // FastGeom::rot: M_k R_n ... R_1
    double last[9];   // M_k: Rotations::m[n] of the exact chain
    float rot32[9];   // Fast32Geom::rot
    int enabled;      // FastGeom::enabled
    int enabled32;    // Fast32Geom::enabled
};

constexpr int kFramesPerLaunch = 128;

struct FramesArgs {
    OutGeom out;
    SrcGeom src;
    Rotations rot;   // n + 1 rotations: the plan's, then a slot for the frame's own
    FastGeom fast;   // the constants all frames share (rot, enabled: per frame)
    const unsigned char* src_px;
    unsigned char* dst_px;
    long long src_frame_stride, dst_frame_stride;  // bytes
    int px_bytes;    // P = channels x element bytes
    int vec;         // gather word: 1, 2, 4, 8 or 16 bytes
    int words;       // NW = P / VEC (<= 4)
    int elem_type;   // double-fisheye source: PB_ELEM_* of its blend (uint8: blend_u8)
    FrameRotation frame[kFramesPerLaunch];
};
static_assert(sizeof(FramesArgs) <= 32764, "kernel parameters are limited to 32764 bytes");

template <int VEC> struct FrameWord { typedef typename WideWord<VEC>::T T; };
template <> struct FrameWord<1> { typedef unsigned char T; };

// One frame of a tile, camera / equirect source: xys[r][c] = source index of tile pixel (r, c);
// warp w stores rows w, w + 8, ..., w + 56 (remap_wide_kernel's gather for one frame).
template <int VEC>
__device__ __forceinline__ void gather_frame_tile(const FramesArgs& a, const int (*xys)[kTileW + 1],
                                                  const unsigned char* __restrict__ sp, unsigned char* __restrict__ dp,
                                                  int row0, int w, int lane) {
    typedef typename FrameWord<VEC>::T Word;
    constexpr int kMaxWords = VEC == 16 ? 2 : kWideMaxWords;  // (P <= 32)
    const int nw = a.words, P = a.px_bytes;
    const long long src_row = (long long)a.src.W * P, dst_row = (long long)a.out.W * P;
#pragma unroll
    for (int g = 0; g < kWideRowsPerWarp; g += kWideRowsInFlight) {
        Word v[kWideRowsInFlight][kMaxWords];
#pragma unroll
        for (int u = 0; u < kWideRowsInFlight; ++u) {
            const int r = w + 8 * (g + u);
            const int xy = row0 + r < a.out.H ? xys[r][lane] : kNoPixel;
            const int at = max(xy, 0);
            const Word* s = reinterpret_cast<const Word*>(sp + (at >> 16) * src_row + (at & 0xffff) * P);
#pragma unroll
            for (int n = 0; n < kMaxWords; ++n) v[u][n] = (n < nw && xy >= 0) ? __ldg(s + n) : Word{};
        }
#pragma unroll
        for (int u = 0; u < kWideRowsInFlight; ++u) {
            const int t = g + u;
            if (row0 + w + 8 * t >= a.out.H) break;
            Word* d = reinterpret_cast<Word*>(dp + 8 * t * dst_row);
#pragma unroll
            for (int n = 0; n < kMaxWords; ++n)
                if (n < nw) d[n] = v[u][n];
        }
    }
}

template <int OUT_KIND, int SRC_KIND>
__global__ void __launch_bounds__(256, PB_WIDE_MIN_CTAS) remap_frames_kernel(const __grid_constant__ FramesArgs a) {
    constexpr bool DBL = SRC_KIND == PB_KIND_DOUBLE;
    __shared__ FastGeom fast;
    __shared__ Rotations rot;
    __shared__ int xys[DBL ? 1 : kTileH][kTileW + 1];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const FrameRotation& fr = a.frame[blockIdx.z];

    // ---------------------------------------------------------------- 0. this frame's constants
    const int n = a.rot.n - 1;  // the plan's rotations; slot n is the frame's own
    {
        const unsigned* s = reinterpret_cast<const unsigned*>(&a.fast);
        unsigned* d = reinterpret_cast<unsigned*>(&fast);
        for (int k = tid; k < (int)(sizeof(FastGeom) / 4); k += blockDim.x) d[k] = s[k];
        for (int k = tid; k < 9 * n; k += blockDim.x) rot.m[k / 9][k % 9] = a.rot.m[k / 9][k % 9];
        if (tid < 9) rot.m[n][tid] = fr.last[tid];
        if (tid == 0) rot.n = a.rot.n;
    }
    __syncthreads();
    if (tid < 9) {
        fast.rot[tid] = fr.rot[tid];
        fast.f32.rot[tid] = fr.rot32[tid];
    }
    if (tid == 0) {
        fast.enabled = fr.enabled;
        fast.f32.enabled = fr.enabled32;
    }
    __syncthreads();

    const int row0 = blockIdx.y * kTileH, col0 = blockIdx.x * kTileW;
    const int rq = tid >> 3, cq = 4 * (tid & 7);  // quad: pixels (rq + 32 q, cq + k), q < 2, k < 4
    const unsigned char* __restrict__ sp = a.src_px + blockIdx.z * a.src_frame_stride;
    unsigned char* __restrict__ dp = a.dst_px + blockIdx.z * a.dst_frame_stride;

    if constexpr (DBL) {
        // ---------------------------------------------------------------- resolve + blend in place
        const int C = a.src.C;
#pragma unroll 1
        for (int q = 0; q < kRowsPerThread; ++q) {
            const int i = row0 + rq + q * kRowGroups;
            if (i >= a.out.H) break;
#pragma unroll 1
            for (int k = 0; k < 4; ++k) {
                const int j = col0 + cq + k;
                if (j >= a.out.W) break;
                const Lookup L = resolve_lookup<OUT_KIND, SRC_KIND>(a.out, fast, rot, a.src, i, j);
                const int off0 = xy_to_offset(L.xy0, a.src.W), off1 = xy_to_offset(L.xy1, a.src.W);
                if (a.elem_type != PB_ELEM_UINT8) {
                    const int P = a.px_bytes;
                    blend_px_typed(off0 >= 0 ? sp + (long long)off0 * P : nullptr, L.w0,
                                   off1 >= 0 ? sp + (long long)off1 * P : nullptr, L.w1,
                                   dp + ((long long)i * a.out.W + j) * P, C, a.elem_type);
                    continue;
                }
                const unsigned char* p0 = sp + (long long)max(off0, 0) * C;
                const unsigned char* p1 = sp + (long long)max(off1, 0) * C;
                unsigned char* o = dp + ((long long)i * a.out.W + j) * C;
                for (int c = 0; c < C; ++c) {
                    const unsigned v0 = off0 >= 0 ? __ldg(p0 + c) : 0u;
                    const unsigned v1 = off1 >= 0 ? __ldg(p1 + c) : 0u;
                    o[c] = blend_u8(v0, L.w0, v1, L.w1);
                }
            }
        }
    } else {
        // ---------------------------------------------------------------- 1. resolve
        unsigned pend = 0;  // bit p: pixel p of this thread is left to the float64 tiers
#pragma unroll 1
        for (int q = 0; q < kRowsPerThread; ++q) {
            const int i = row0 + rq + q * kRowGroups;
#pragma unroll 4
            for (int k = 0; k < 4; ++k) {
                const int p = q * 4 + k, j = col0 + cq + k;
                int xy = kNoPixel;
                if (i < a.out.H && j < a.out.W) {
                    Lookup L;
                    if (fast.f32.enabled && fast32_lookup<OUT_KIND, SRC_KIND>(a.out, fast.f32, a.src, i, j, L)) xy = L.xy0;
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
                xys[r][c] = resolve_lookup64<OUT_KIND, SRC_KIND>(a.out, fast, rot, a.src, row0 + r, col0 + c).xy0;
            }
        }
        __syncthreads();

        // ---------------------------------------------------------------- 2. gather
        const int j = col0 + lane;
        if (j >= a.out.W) return;
        unsigned char* const d0 = dp + ((long long)(row0 + w) * a.out.W + j) * a.px_bytes;
        switch (a.vec) {
            case 16: gather_frame_tile<16>(a, xys, sp, d0, row0, w, lane); break;
            case 8: gather_frame_tile<8>(a, xys, sp, d0, row0, w, lane); break;
            case 4: gather_frame_tile<4>(a, xys, sp, d0, row0, w, lane); break;
            case 2: gather_frame_tile<2>(a, xys, sp, d0, row0, w, lane); break;
            default: gather_frame_tile<1>(a, xys, sp, d0, row0, w, lane); break;
        }
    }
}

}  // namespace pb
