// pb_boxes.cuh -- the two tile classes of a batch through a double-fisheye source, staged box by box
// and fed by a producer warp.
//
// The batched kernels of pb_tiled.cuh / pb_tiled2.cuh stage the bounding rectangle of a tile's
// footprint in 16-row TMA boxes.  A footprint runs diagonally through the source, so that rectangle
// is ~3x the bytes the tile reads; giving each box its own first column and width cuts the staged
// bytes by a quarter (tests/analysis/stair_sim.py).  The extents are a property of the geometry:
// pb_box_kernel records them once per plan.
//
// Issuing boxes of different widths costs the issuing thread a table read per box; with thread 0 of
// a consumer warp doing it, the whole block waited for that warp at every frame's barrier
// (profiles/experiments/README.md, staircase of boxes).  Here one extra warp per CTA does all TMA
// traffic -- box loads, group refills, tile stores -- and the consumer warps never meet at a block
// barrier inside the frame loop.  Three kinds of mbarrier connect them:
//   full[g]     frame group g holds its frame (TMA transaction count, armed by the producer)
//   empty[g]    every consumer thread has gathered from group g and written (and fenced) its quads
//               of the frame's output tile: the producer refills g and stores the tile
//   outfree[b]  the store of output tile b has finished reading it (after wait_group.read)
// The float64 operations of the resolve and their order are those of the other batched kernels:
// only the integer offset of a pixel inside its frame group changes, so the output is bit-identical.
#pragma once

#include "pb_tiled2.cuh"

namespace pb {

constexpr int kMaxBoxes = 8;  // boxes per (tile, slot) the table describes: footprints of up to 128 source rows

// Per-box extents of every (tile, slot) footprint of a separable double-fisheye plan, one warp per
// tile.  Entry (tile, slot, k), k < kMaxBoxes, is {first staged byte of the box's rows (16-byte
// aligned, TMA), width in 16-byte units (odd: names one of the plan's tensor maps; 0: nothing to
// stage), byte offset of the box inside a frame group (after its 128 zero bytes), first source row}.
// Boxes are laid out slot 0 first, then slot 1, each 16 rows of 16 * width bytes.  A tile whose
// footprint needs more than kMaxBoxes boxes has width -1 in every entry.
// Every pixel is resolved with the operations of the kernels' resolve step (same truncations, same
// in-image test), so each box holds exactly the columns its rows reference.
__global__ void __launch_bounds__(256) pb_box_kernel(const __grid_constant__ TiledArgs a, const int4* __restrict__ tile_fp,
                                                     int4* __restrict__ boxes, int tiles_x, int n_tiles) {
    __shared__ int mn[8][kMaxBoxes], mx[8][kMaxBoxes];
    const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x * 8 + wp;
    if (tile >= n_tiles) return;
    const int x0 = (tile % tiles_x) * kTileW, y0 = (tile / tiles_x) * kTileH;
    const double2 cs = __ldg(reinterpret_cast<const double2*>(a.col_tab) + min(x0 + lane, a.out.W - 1));
    int xb[2], units[2], row[2];
    bool described = true;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int4 fp = tile_fp[2 * tile + s];
        const int nbox = fp.z;
        if (nbox > kMaxBoxes) described = false;
        if (lane < kMaxBoxes) {
            mn[wp][lane] = 0x7fffffff;
            mx[wp][lane] = -1;
        }
        __syncwarp();
        const int w = s ? a.src.wr : a.src.wl;
        const double cx = s ? a.src.cxr : a.src.cxl;
        const bool all_valid = fp.w & 1;
        bool outside = false;  // a pixel outside the footprint's rows: stage the rectangle instead
        if (nbox > 0 && nbox <= kMaxBoxes) {
            for (int r = 0; r < kTileH; ++r) {
                const double d = __ldg(a.row_tab + 4 * min(y0 + r, a.out.H - 1) + s);
                double fx, fy;
                camera_fxy(cs.x, cs.y, d, a.src.cy, cx, fx, fy);
                if (!(all_valid || inside_image(fx, fy, w, a.src.H))) continue;
                int px = trunc_abs(fx);
                if (s) px = a.src.W - 1 - px;
                const int k = (trunc_abs(fy) - fp.x) >> 4;
                if (k < 0 || k >= nbox) {
                    outside = true;
                    continue;
                }
                atomicMin(&mn[wp][k], px);
                atomicMax(&mx[wp][k], px);
            }
        }
        outside = __any_sync(0xffffffffu, outside);
        __syncwarp();
        xb[s] = 0;
        units[s] = 0;
        row[s] = fp.x + lane * kBoxRows;
        if (lane < nbox && lane < kMaxBoxes) {  // (a tile of more boxes is not described: see below)
            if (outside) {
                xb[s] = fp.y;
                units[s] = stage_units(fp.w >> 1);
            } else if (mx[wp][lane] >= 0) {
                xb[s] = (mn[wp][lane] * 3) & ~15;
                units[s] = stage_units(mx[wp][lane] * 3 + 3 - xb[s]);
            }
        }
        __syncwarp();
    }
    // byte offsets inside a frame group: an exclusive scan over slot 0's boxes, then slot 1's
    int goff[2];
    int base = 0;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        int incl = lane < kMaxBoxes ? kBoxRows * 16 * units[s] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        goff[s] = base + incl - (lane < kMaxBoxes ? kBoxRows * 16 * units[s] : 0);
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane < kMaxBoxes) {
#pragma unroll
        for (int s = 0; s < 2; ++s)
            boxes[((size_t)tile * 2 + s) * kMaxBoxes + lane] =
                described ? make_int4(xb[s], units[s], goff[s], row[s]) : make_int4(0, -1, 0, 0);
    }
}

// Shared state of a CTA of remap_boxes_kernel (after the output tiles and the ring of frame groups)
struct alignas(16) BoxShared {
    uint64_t full[kMaxGroups];
    uint64_t empty[kMaxGroups];
    uint64_t outfree[2];
    int2 box[2 * kMaxBoxes];  // per (slot, box): {row pitch, offset constant}: a pixel at source row y and
                              // byte column xb sits at y * pitch + xb + constant inside its frame group
};

// CLS 1: tiles that see one lens at unit weights, 256 consumer threads (two quads each), 4 CTAs per SM.
// CLS 2: tiles that see both lenses or the blend band, 512 consumer threads (one quad each), 2 CTAs per SM.
template <int CLS>
struct BoxKernel {
    static constexpr int kConsumers = CLS == 1 ? kTileThreads : kTile2Threads;
    static constexpr int kThreads = kConsumers + 32;  // + the producer warp
    static constexpr int kMinCtas = CLS == 1 ? 4 : 2;
    static constexpr int kRows = kTileH * kQuadsPerRow / kConsumers;  // quads (rows) per consumer thread
    static constexpr int kRowStep = kConsumers / kQuadsPerRow;        // rows between a thread's quads
    static constexpr int kSlots = CLS == 1 ? 1 : 2;
};

template <int CLS>
__global__ void __launch_bounds__(BoxKernel<CLS>::kThreads, BoxKernel<CLS>::kMinCtas)
remap_boxes_kernel(const __grid_constant__ TiledArgs a) {
    using K = BoxKernel<CLS>;
    constexpr int NS = K::kSlots, RPT = K::kRows;
    extern __shared__ __align__(128) unsigned char smem[];
    // [ out tiles: 2 x 6144 ][ ring of frame groups: stage_bytes + 128 ][ BoxShared ]
    unsigned char* out_tiles = smem;
    unsigned char* stages = smem + 2 * kOutTileBytes;
    BoxShared* sh = reinterpret_cast<BoxShared*>(stages + a.stage_bytes + 128);

    const int tid = threadIdx.x;
    const bool producer = tid >= K::kConsumers;
    const int qc = tid & (kQuadsPerRow - 1);
    const int rg = tid >> 3;
    int tile_x, tile_y;
    {
        const int t = __ldg(a.tile_list + blockIdx.x);
        tile_y = t / a.tiles_x;
        tile_x = t - tile_y * a.tiles_x;
    }
    const int tile = tile_y * a.tiles_x + tile_x;
    const int x0 = tile_x * kTileW;
    const int y0 = tile_y * kTileH;

    if (tid == 0) {
        ptx::prefetch_tensormap(&a.dst_map);
#pragma unroll
        for (int g = 0; g < kMaxGroups; ++g) {
            ptx::mbarrier_init(&sh->full[g], 1);
            ptx::mbarrier_init(&sh->empty[g], K::kConsumers);
        }
        ptx::mbarrier_init(&sh->outfree[0], 1);
        ptx::mbarrier_init(&sh->outfree[1], 1);
        ptx::fence_mbarrier_init();
    }

    // ------------------------------------------------------------ footprints, boxes, tables
    const int4 f0 = __ldg(a.tile_fp + 2 * tile), f1 = __ldg(a.tile_fp + 2 * tile + 1);
    const int4* __restrict__ bt = a.tile_box + (size_t)tile * 2 * kMaxBoxes;
    // the last entry ends the frame group (boxes are laid out in entry order)
    const int4 last = __ldg(bt + 2 * kMaxBoxes - 1);
    const int group_bytes = 128 + last.z + kBoxRows * 16 * last.y;
    // (CLS 1: the tile's one lens is slot 0 of the kernel)
    const bool right_lens = CLS == 1 && f0.z == 0;
    int4 fpv[NS];
    fpv[0] = right_lens ? f1 : f0;
    if (NS == 2) fpv[NS - 1] = f1;
    bool wide = last.y < 0;
#pragma unroll
    for (int s = 0; s < NS; ++s)
        if (fpv[s].z > 0 && stage_units(fpv[s].w >> 1) > a.max_units) wide = true;
    const int n_groups = min(min(kMaxGroups, a.n_frames), (a.stage_bytes + 128) / group_bytes);
    if (wide || n_groups < 1) {  // block-uniform: a footprint that cannot be staged (a pole)
        direct_tile<PB_KIND_EQUIRECT, PB_KIND_DOUBLE, 1>(a, nullptr, nullptr, out_tiles, x0, y0);
        return;
    }
    int4 mybox = make_int4(0, 0, 0, 0);  // producer lane j < 2 * kMaxBoxes: box j of the table
    if (tid < 2 * kMaxBoxes || (producer && tid - K::kConsumers < 2 * kMaxBoxes)) {
        const int j = producer ? tid - K::kConsumers : tid;
        mybox = __ldg(bt + j);
        if (!producer) {
            const int pitch = 16 * mybox.y;
            sh->box[j] = make_int2(pitch, 128 + mybox.z - mybox.w * pitch - mybox.x);
        }
    }
    if (tid < n_groups * 8) reinterpret_cast<int4*>(stages + (tid >> 3) * group_bytes)[tid & 7] = make_int4(0, 0, 0, 0);

    const unsigned stages_sa = ptx::smem_addr(stages);
    if (producer) {
        (void)__syncthreads_and(true);  // barriers initialised (the consumers' barrier below)
        const int lane = tid - K::kConsumers;
        // CLS 1: only the boxes of the tile's lens hold anything (the other slot's are 0 units wide)
        const bool mine = lane < 2 * kMaxBoxes && mybox.y > 0;
        const CUtensorMap* map = &a.src_maps[mine ? (mybox.y - kMinStageUnits) >> 1 : 0];
        const uint64_t keep = ptx::policy_of(a.load_policy);
        const uint64_t drop = ptx::policy_of(a.store_policy);
        auto issue_group = [&](int f, int g) {  // the whole warp: every box of frame f into group g
            if (lane == 0) ptx::mbarrier_arrive_expect_tx(&sh->full[g], (unsigned)(group_bytes - 128));
            __syncwarp();
            if (mine)
                ptx::tma_load_3d_hint(stages + g * group_bytes + 128 + mybox.z, map, mybox.x >> 1, mybox.w, f, &sh->full[g],
                                      keep);
        };
        for (int f = 0; f < n_groups; ++f) issue_group(f, f);
        const unsigned empty_sa = ptx::smem_addr(&sh->empty[0]);
        const int ys = y0 - a.tile_y0 * kTileH;
        int g = 0;
        unsigned parity = 0;
        for (int f = 0; f < a.n_frames; ++f) {
            ptx::mbarrier_wait_sa(empty_sa + 8 * g, parity);  // frame f is gathered and its tile written
            if (f + n_groups < a.n_frames) issue_group(f + n_groups, g);
            if (lane == 0) {
                ptx::tma_store_3d_hint(&a.dst_map, x0 * 3, ys, f, out_tiles + (f & 1) * kOutTileBytes, drop);
                ptx::bulk_commit();
                ptx::bulk_wait_read0();
                ptx::mbarrier_arrive(&sh->outfree[f & 1]);
            }
            __syncwarp();
            if (++g == n_groups) {
                g = 0;
                parity ^= 1u;
            }
        }
        return;
    }

    // ------------------------------------------------------------ consumers: resolve once per tile
    double2 cs[4];
    {
        const double2* __restrict__ col = reinterpret_cast<const double2*>(a.sep1_col) + tile_x * kTileW;
#pragma unroll
        for (int k = 0; k < 4; ++k) cs[k] = __ldg(col + k * 8 + qc);
    }
    double2 r01[RPT], wrow[RPT];
#pragma unroll
    for (int q = 0; q < RPT; ++q) {
        const double2* __restrict__ row = reinterpret_cast<const double2*>(a.sep1_row) + 2 * (y0 + rg + q * K::kRowStep);
        r01[q] = __ldg(row);
        wrow[q] = (CLS == 2) ? __ldg(row + 1) : make_double2(1.0, 1.0);
    }
    // CLS 2: is every blend weight of the tile exactly 1?  (also: barriers, box constants and zero bytes visible)
    bool unit = true;
#pragma unroll
    for (int q = 0; q < RPT; ++q) unit = unit && wrow[q].x == 1.0 && wrow[q].y == 1.0;
    const bool unit_weights = __syncthreads_and(unit);

    unsigned adr[NS][4 * RPT], shf[NS][4 * RPT];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const bool right = CLS == 1 ? right_lens : s != 0;
        const int bs = right ? kMaxBoxes : 0;  // the slot's boxes in the table
        const int w = right ? a.src.wr : a.src.wl;
        const double cx = right ? a.src.cxr : a.src.cxl;
#pragma unroll
        for (int q = 0; q < RPT; ++q) {
            const double dist = right ? r01[q].y : r01[q].x;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                unsigned rel = 0;  // the group's zero bytes: no source pixel
                if (fpv[s].z > 0) {
                    double fx, fy;
                    camera_fxy(cs[k].x, cs[k].y, dist, a.src.cy, cx, fx, fy);
                    int px = trunc_abs(fx);
                    if (right) px = a.src.W - 1 - px;
                    const int py = trunc_abs(fy);
                    const int2 b = sh->box[bs + (((py - fpv[s].x) >> 4) & (kMaxBoxes - 1))];
                    if ((fpv[s].w & 1) || inside_image(fx, fy, w, a.src.H)) rel = (unsigned)(py * b.x + px * 3 + b.y);
                }
                adr[s][q * 4 + k] = stages_sa + (rel & ~3u);
                shf[s][q * 4 + k] = rel << 3;
            }
        }
    }
    // blend of each row of this thread: 0 = unit weights (exact byte add), 1 = guarded fixed point, 2 = float64
    unsigned wfix[RPT][2];
    int wmode[RPT];
#pragma unroll
    for (int q = 0; q < RPT; ++q) {
        wfix[q][0] = wfix[q][1] = 0;
        wmode[q] = 0;
        if (CLS == 2 && !unit_weights && !(wrow[q].x == 1.0 && wrow[q].y == 1.0))
            wmode[q] = fix_weights(wrow[q].x, wrow[q].y, wfix[q][0], wfix[q][1]) ? 1 : 2;
    }

    // ------------------------------------------------------------ consumers: frame loop
    const unsigned out_sa = ptx::smem_addr(out_tiles) + rg * kOutRowBytes + qc * 12;
    const unsigned full_sa = ptx::smem_addr(&sh->full[0]);
    const unsigned outfree_sa = ptx::smem_addr(&sh->outfree[0]);
    const unsigned empty_sa = ptx::smem_addr(&sh->empty[0]);
    constexpr bool DENSE = CLS == 2;
    auto frame_loop = [&](auto ACT, auto WGT) {
        constexpr int act = decltype(ACT)::value;   // 1: slot 0 only, 2: slot 1 only, 3: both
        constexpr bool wgt = decltype(WGT)::value;  // some row of the tile has a weighted blend
        int g = 0;
        unsigned parity = 0;
        for (int f = 0; f < a.n_frames; ++f) {
            const unsigned goff = (unsigned)(g * group_bytes);
            ptx::mbarrier_wait_sa(full_sa + 8 * g, parity);
            unsigned v[4 * RPT], w[4 * RPT];
#pragma unroll
            for (int p = 0; p < 4 * RPT; ++p) {
                v[p] = (act & 1) ? lean_pick<DENSE>(adr[0][p], goff, shf[0][p]) : 0u;
                w[p] = (act & 2) ? lean_pick<DENSE>(adr[NS - 1][p], goff, shf[NS - 1][p]) : 0u;
            }
#pragma unroll
            for (int q = 0; q < RPT; ++q) {
                if (!wgt || wmode[q] == 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int p = q * 4 + k;
                        v[p] = (act == 3) ? __vadd4(v[p], w[p]) : (act == 1 ? v[p] : w[p]);
                    }
                } else if (wmode[q] == 1) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        v[q * 4 + k] = blend_px_fix(v[q * 4 + k], wfix[q][0], wrow[q].x, w[q * 4 + k], wfix[q][1], wrow[q].y);
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) v[q * 4 + k] = blend_px_weighted(v[q * 4 + k], wrow[q].x, w[q * 4 + k], wrow[q].y);
                }
            }
            // the store of frame f - 2 has left this output tile
            ptx::mbarrier_wait_sa(outfree_sa + 8 * (f & 1), ((unsigned)(f >> 1) & 1u) ^ 1u);
            const unsigned o = out_sa + (f & 1) * kOutTileBytes;
#pragma unroll
            for (int q = 0; q < RPT; ++q) store_quad_sa(o + q * K::kRowStep * kOutRowBytes, v + q * 4);
            ptx::fence_async_smem();
            ptx::mbarrier_arrive_sa(empty_sa + 8 * g);
            if (++g == n_groups) {
                g = 0;
                parity ^= 1u;
            }
        }
    };
    const int n_act = (fpv[0].z > 0) + (NS == 2 && fpv[NS - 1].z > 0);
    if (CLS == 1 || unit_weights) {
        if (n_act == 2) frame_loop(std::integral_constant<int, 3>{}, std::false_type{});
        else if (NS == 1 || fpv[NS - 1].z == 0) frame_loop(std::integral_constant<int, 1>{}, std::false_type{});
        else frame_loop(std::integral_constant<int, 2>{}, std::false_type{});
    } else {
        if (n_act == 2) frame_loop(std::integral_constant<int, 3>{}, std::true_type{});
        else if (fpv[NS - 1].z == 0) frame_loop(std::integral_constant<int, 1>{}, std::true_type{});
        else frame_loop(std::integral_constant<int, 2>{}, std::true_type{});
    }
}

inline int boxes_smem_bytes(int stage_bytes) {
    return 2 * kOutTileBytes + stage_bytes + 128 + (int)sizeof(BoxShared) + 128;
}

}  // namespace pb
