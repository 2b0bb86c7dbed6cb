// pt_mega.cuh — single-launch "megakernels".
//
//  k_mega_pixel : base / lmem / grid variants.  One thread per pixel runs the pixel's whole sample
//                 sequence (the per-pixel RNG stream makes samples of one pixel inherently serial,
//                 SURVEY.md 0.3); a warp covers an 8x4 pixel tile so its 32 rays stay coherent.
//                 Replaces kernel pathTracer of base:220-241, lmem:218-254, grid:348-381.
//  k_mega_nodof : CLSuperPathTracer_lmem_NoDoF.  The reference launches 64 work-items per pixel, writes a
//                 268 MB float4 scratch image and reduces it with a second kernel (nodof:217-274).
//                 Here one warp owns one pixel: lane l traces samples l and l+32, adds them (tree level
//                 32), and five shuffle-down steps finish the reference's exact reduction tree in
//                 registers — no scratch image, no second launch, same float sums.
#pragma once
#include <time.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "pt_host.h"

// 1: the big-grid megakernel inlines TraceRay twice (sample_two_traces).  Round 1 measured that form faster at the 64-register budget
// (4.57 vs 4.77 ms per 4 spp); with the leaner grid walk of round 2 the single ray loop wins (12.29 vs 12.57 ms per 16 spp).
#ifndef PT_BIG_TWO_TRACES
#define PT_BIG_TWO_TRACES 0
#endif
namespace pt {

__constant__ SceneBlock c_scene;

// Stage the used part of the scene block from global into shared memory (the _lmem idea, lmem:232-244,
// without its "work-group must be at least ntriangles big" limitation): ONE bulk asynchronous copy (TMA,
// cp.async.bulk -> UBLKCP) issued by thread 0 and an mbarrier the whole CTA waits on, instead of a
// load/store loop through registers.
PT_DEV const SceneBlock *stage_scene_smem(const LaunchArgs &P, unsigned char *smem) {
    __shared__ __align__(8) uint64_t s_stage_bar;
    if (threadIdx.x == 0) {
        mbar_init(&s_stage_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(&s_stage_bar, (uint32_t)P.scene_bytes);
        tma_load_1d(smem, P.gscene, (uint32_t)P.scene_bytes, &s_stage_bar);
    }
    mbar_wait(&s_stage_bar, 0);
    return reinterpret_cast<const SceneBlock *>(smem);
}

// Work counters: warp shuffle-reduce, then native 32-bit shared-memory atomics per warp (a 64-bit shared atomicAdd
// is a compare-and-swap loop: it was 6 % of the NoDoF kernel's instructions), then ONE set of 64-bit global atomics
// per CTA (none for zero sums) — the wavefront kernels call this once per launch, so per-warp atomics on seven
// global addresses would serialise in L2.  Per-CTA raw sums fit 32 bits (<= 1024 threads x u32 per-thread counters
// that themselves stay far below 2^22 here); the products with the triangle / primitive counts are formed in 64 bits.
// Must be reached by every thread of the CTA.
PT_DEV void flush_counters(const LaunchArgs &P, const Counters &c, int ntri_counted, int nprims) {
    __shared__ unsigned int s_raw[6];          // samples rays shadow cells gtri btests
    if (threadIdx.x < 6) s_raw[threadIdx.x] = 0u;
    __syncthreads();
    uint32_t rays = __reduce_add_sync(0xffffffffu, c.rays);
    uint32_t shadow = __reduce_add_sync(0xffffffffu, c.shadow);
    uint32_t cells = __reduce_add_sync(0xffffffffu, c.cells);
    uint32_t gtri = __reduce_add_sync(0xffffffffu, c.gtri);
    uint32_t samples = __reduce_add_sync(0xffffffffu, c.samples);
    uint32_t loops = __reduce_add_sync(0xffffffffu, c.btests);
    if ((threadIdx.x & 31) == 0) {
        if (samples) atomicAdd(&s_raw[0], samples);
        if (rays) atomicAdd(&s_raw[1], rays);
        if (shadow) atomicAdd(&s_raw[2], shadow);
        if (cells) atomicAdd(&s_raw[3], cells);
        if (gtri) atomicAdd(&s_raw[4], gtri);
        if (loops) atomicAdd(&s_raw[5], loops);
    }
    __syncthreads();
    if (threadIdx.x < 7 && P.counters) {
        const unsigned long long r = s_raw[1], g = s_raw[4];
        unsigned long long v;
        switch (threadIdx.x) {
            case 0: v = s_raw[0]; break;                                             // samples
            case 1: v = r; break;                                                    // rays
            case 2: v = s_raw[2]; break;                                             // shadow rays
            case 3: v = g + r * (unsigned long long)ntri_counted; break;             // tri_tests (nominal)
            case 4: v = s_raw[3]; break;                                             // cells visited
            case 5: v = r * (unsigned long long)nprims; break;                       // prim_tests
            default: v = s_raw[5]; break;                                            // tri_tests executed (after the conservative culls)
        }
        if (v) atomicAdd(P.counters + threadIdx.x, v);
    }
}

// The state a pixel's sample loop carries from one sample to the next is its colour sum and its RNG state, nothing else.
// A launch starts it fresh (seeded from the pixel id, the bias c0) or, continuing a progression, where the previous
// range of it left the pixel.  Read once, before the sample loop.
PT_DEV void pixel_state_in(const LaunchArgs &P, uint32_t pix, Rng &rng, float &cx, float &cy, float &cz) {
    if (P.rng_in) {
        const uint4 r = P.rng_in[pix];
        const float4 a = P.accum_in[pix];
        rng.x0 = r.x; rng.x1 = r.y; rng.c0 = r.z; rng.c1 = r.w;
        cx = a.x; cy = a.y; cz = a.z;
    } else {
        rng = rng_seed(P.seeds, pix);
        cx = cy = cz = P.c0;
    }
}

// convert_uchar4 of the colour sum (or, on a range that does not end the frame, of the preview ((c - 13) * f) + 13 with
// f = spp / samples done, each operation rounded on its own), plus the optional float buffer and final RNG state.  The
// thread that read the pixel's state writes it, so input and output of a range may be the same buffers.
PT_DEV void pixel_state_out(const LaunchArgs &P, size_t pix, const Rng &rng, float cx, float cy, float cz) {
    if (P.preview != 0.0f) {
        const float f = P.preview;
        P.rgba[pix] = pack_rgba8_rz(__fadd_rn(__fmul_rn(__fsub_rn(cx, 13.0f), f), 13.0f), __fadd_rn(__fmul_rn(__fsub_rn(cy, 13.0f), f), 13.0f),
                                    __fadd_rn(__fmul_rn(__fsub_rn(cz, 13.0f), f), 13.0f), P.alpha);
    } else {
        P.rgba[pix] = pack_rgba8_rz(cx, cy, cz, P.alpha);
    }
    if (P.accum) P.accum[pix] = make_float4(cx, cy, cz, P.alpha);
    if (P.rng_out) P.rng_out[pix] = make_uint4(rng.x0, rng.x1, rng.c0, rng.c1);
}

// BIG, trianglegrid: grids whose records do not stay in L1 — 64 registers / 8 CTAs per SM (72 / 7: 14.78 vs 14.51 ms per 16 spp)
// and the longest-tile-first launch order; otherwise 80 registers / 6 CTAs.  Both use the single ray loop (PT_BIG_TWO_TRACES).
// BIG, brute-force variants: frames above 400 k pixels — per-cluster triangle culling compiled in (tri_loop<.., CL>).
// Measured (B200): soup 1 M triangles 4.57 ms per 4 spp with BIG vs 4.87 without; default 96-triangle grid scene
// 1.41 ms without vs 1.58 with.
template <int VARIANT, bool FMA, int MEM, bool BIG>
__global__ void __launch_bounds__(128, (BIG && VARIANT == PT_VARIANT_GRID) ? 8 : 6) k_mega_pixel(const __grid_constant__ LaunchArgs P) {
    constexpr bool CARRY = VARIANT != PT_VARIANT_BASE;
    constexpr bool GRID = VARIANT == PT_VARIANT_GRID;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SceneBlock *S = (MEM == PT_SCENE_SMEM) ? stage_scene_smem(P, smem_raw) : &c_scene;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long t_start = 0;
    if (BIG && P.cta_times && threadIdx.x == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_start));
    // tile of this CTA: its 2-D block index, or — 1-D launches of the big-grid kernel — entry blockIdx.x of the launch order
    // (longest tile first, see launch_pixel_b)
    uint32_t bx = blockIdx.x, by = blockIdx.y;
    if (BIG && P.tile_order) {
        const uint32_t tile = __ldg(P.tile_order + blockIdx.x);
        by = tile / P.tiles_x; bx = tile - by * P.tiles_x;
    }
    // 4 warps: 16x8 pixel tile (2x2 warps of 8x4 pixels); 2 warps: 16x4; 1 warp: 8x4 (launch_pixel_b picks the block size)
    const int tw = blockDim.x >= 64 ? 2 : 1, th = (int)(blockDim.x >> 5) / tw;
    const int i = bx * (8 * tw) + (warp % tw) * 8 + (lane & 7);
    const int vr = by * (4 * th) + (warp / tw) * 4 + (lane >> 3);
    Counters cnt = {0, 0, 0, 0, 0, 0};
    const int j = map_row(P, vr);
    if (i < P.W && vr < P.nrows && j < P.row_end) {
        Rng rng;
        float cx, cy, cz;
        pixel_state_in(P, (uint32_t)(j * P.W + i), rng, cx, cy, cz);
        for (int s = 0; s < P.spp; ++s) {
            V3 o, d;
            camera_ray<FMA>(P.cam, rng, i, j, o, d);
            V3 c = (BIG && GRID && PT_BIG_TWO_TRACES) ? sample_two_traces<FMA, CARRY, GRID>(P.ap, S, P.grid, o, d, rng, cnt)
                                 : sample<FMA, CARRY, GRID, BIG && !GRID>(P.ap, S, P.grid, o, d, rng, cnt);
            cx = Ar<FMA>::madd(c.x, P.scale, cx);
            cy = Ar<FMA>::madd(c.y, P.scale, cy);
            cz = Ar<FMA>::madd(c.z, P.scale, cz);
        }
        pixel_state_out(P, (size_t)j * P.W + i, rng, cx, cy, cz);
    }
    if (GRID) cnt.btests = cnt.gtri;        // trace_grid tests every record of the cells it visits
    flush_counters(P, cnt, GRID ? 0 : S->ntri_counted, P.ap.nsq + P.ap.nsp);
    if (BIG && P.cta_times && threadIdx.x == 0) {
        unsigned long long t_end;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_end));
        const size_t b = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
        P.cta_times[2 * b] = t_start; P.cta_times[2 * b + 1] = t_end;
    }
}

template <bool FMA, int MEM>     // 8 warps = a 4x2 pixel tile per CTA (4x1 tiles time the same, 2x1 tiles 3 % slower)
__global__ void __launch_bounds__(256, 4) k_mega_nodof(const __grid_constant__ LaunchArgs P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SceneBlock *S = (MEM == PT_SCENE_SMEM) ? stage_scene_smem(P, smem_raw) : &c_scene;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = blockIdx.x * 4 + (warp & 3);
    const int vr = blockIdx.y * 2 + (warp >> 2);
    Counters cnt = {0, 0, 0, 0, 0, 0};
    const int py = map_row(P, vr);
    // (a grid-stride persistent form of this kernel — one resident wave of CTAs, warps striding over the pixels — was
    // measured slower: 0.434 ms vs 0.409 ms; the hardware CTA scheduler balances the uneven pixels better)
    if (px < P.W && vr < P.nrows && py < P.row_end) {   // warp-uniform
        float ax = 0.f, ay = 0.f, az = 0.f, bx = 0.f, by = 0.f, bz = 0.f;
#pragma unroll 1                                                    // ONE copy of Sample(): the code stays i-cache resident
        for (int h = 0; h < 2; ++h) {
            const int li = lane + 32 * h;                       // local id inside the 8x8 group
            const int gi = 8 * px + (li & 7), gj = 8 * py + (li >> 3);
            const uint32_t gid = (uint32_t)(gj * (8 * P.W) + gi);
            Rng rng = rng_seed(P.seeds, gid);
            V3 o, d;
            camera_ray<FMA>(P.cam, rng, px, py, o, d);
            V3 c = sample<FMA, true, false>(P.ap, S, P.grid, o, d, rng, cnt);
            if (h == 0) { ax = __fmul_rn(c.x, 3.5f); ay = __fmul_rn(c.y, 3.5f); az = __fmul_rn(c.z, 3.5f); }
            else        { bx = __fmul_rn(c.x, 3.5f); by = __fmul_rn(c.y, 3.5f); bz = __fmul_rn(c.z, 3.5f); }
            if (P.rng_out) P.rng_out[gid] = make_uint4(rng.x0, rng.x1, rng.c0, rng.c1);
        }
        // nodof:253-274 reduction tree: li += li+32, then +16, +8, +4, +2, +1
        float sx = __fadd_rn(ax, bx), sy = __fadd_rn(ay, by), sz = __fadd_rn(az, bz);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            sx = __fadd_rn(sx, __shfl_down_sync(0xffffffffu, sx, off));
            sy = __fadd_rn(sy, __shfl_down_sync(0xffffffffu, sy, off));
            sz = __fadd_rn(sz, __shfl_down_sync(0xffffffffu, sz, off));
        }
        if (lane == 0) {
            sx = __fadd_rn(sx, 13.0f); sy = __fadd_rn(sy, 13.0f); sz = __fadd_rn(sz, 13.0f);
            const size_t pix = (size_t)py * P.W + px;
            P.rgba[pix] = pack_rgba8_rz(sx, sy, sz, 255.0f);
            if (P.accum) P.accum[pix] = make_float4(sx, sy, sz, 255.0f);
        }
    }
    flush_counters(P, cnt, S->ntri_counted, P.ap.nsq + P.ap.nsp);
}

// ---- launch order of the big-grid megakernel's tiles: LONGEST FIRST, from measured CTA durations -----------------------
// A pixel's sample chain is indivisible, so the unit of work is one CTA (16x8 pixels) — 5.1 ms on average, up to 12.9 ms,
// for one rank's stripes of the strong-scaled config-5 frame (3840x2160x64 over 8 ranks), whose whole launch is 6.9 waves
// = 39 ms long.  In raster order the last CTAs start at 32.5 ms and the launch ramps down for another 8.5 ms: 85.6 % of
// the CTA slot-time is used (98.3 % for the full frame on one GPU) — the 11 % the strong-scaling curve lost at N = 8
// (tools/cta_timeline.py, profiles/r2_09).  The hardware hands out CTAs in block-index order, so the kernel reads its
// tile from a table sorted by COST, longest first (LPT list scheduling): the cheap tiles fill the end of the launch.
// Costs are measured, not guessed: the first launch of a geometry (image size, rows / stripes of this rank, camera, grid)
// runs in raster order while every CTA records its globaltimer span; every later launch of that geometry uses the table
// sorted from those durations.  Which CTA renders which tile never affects results, and a table left over from another
// scene with the same geometry is merely a worse order.  (Tried and dropped: classifying tiles by "primary ray hits the
// grid box" — no gain, floor tiles are as expensive, their shadow rays cross the grid; a 1-spp pre-pass as the cost
// estimate for the FIRST launch — its order was no better than raster, one sample per pixel says too little about 256;
// 1-warp CTAs, to shrink the unit — 3 % slower.)  The key is the geometry, not the sample count: a progression in ranges
// of >= 16 samples (pt_launch_pathtracer_range) records in its first range and runs sorted from its second on, and a
// one-launch frame after it on the same context reuses that order.
struct TileOrderKey {
    int W, H, row_begin, row_end, nrows, stripe_h, rank, nranks, variant_fma, ntri;
    unsigned long long scene_version;
    Camera cam;
    float bmin[3], bmax[3], cell[3];
    int res[3];
};

static double tile_order_now_ms() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec / 1e6;
}

static int tile_order_rebuild(pt_ctx ctx, size_t n, bool identity) {
    const double t0 = tile_order_now_ms();
    PT_CUDA(cudaMemcpyAsync(ctx->h_cta_times, ctx->d_cta_times, n * 16, cudaMemcpyDeviceToHost, ctx->stream), "read CTA times");
    PT_CUDA(cudaStreamSynchronize(ctx->stream), "sync CTA times");
    const double t1 = tile_order_now_ms();
    std::vector<std::pair<unsigned long long, uint32_t>> cost(n);
    for (size_t b = 0; b < n; ++b) {
        const unsigned long long t0 = ctx->h_cta_times[2 * b], t1 = ctx->h_cta_times[2 * b + 1];
        const uint32_t tile = identity ? (uint32_t)b : ctx->h_tile_order[b];
        cost[b] = std::make_pair(t1 > t0 ? t1 - t0 : 0ull, tile);
    }
    std::sort(cost.begin(), cost.end(), [](const std::pair<unsigned long long, uint32_t> &a, const std::pair<unsigned long long, uint32_t> &b) {
        return a.first != b.first ? a.first > b.first : a.second < b.second;
    });
    for (size_t b = 0; b < n; ++b) ctx->h_tile_order[b] = cost[b].second;
    PT_CUDA(cudaMemcpyAsync(ctx->d_tile_order, ctx->h_tile_order, n * 4, cudaMemcpyHostToDevice, ctx->stream), "upload tile order");
    if (getenv("PT_DEBUG_AUTO"))
        fprintf(stderr, "ptcuda: tile order rebuilt for %zu tiles (%s): wait for the GPU %.2f ms, sort %.2f ms\n", n,
                identity ? "first launch, raster order" : "ordered launch", t1 - t0, tile_order_now_ms() - t1);
    return 0;
}

// `other`: another kernel with k_mega_pixel's tiling and launch contract (PT_KERNEL_GRID_QUEUE) to launch in its place
template <int VARIANT, bool FMA, int MEM, bool BIG>
static int launch_pixel_b(pt_ctx ctx, const LaunchArgs &args_in, void (*other)(const LaunchArgs) = nullptr) {
    void (*kern)(const LaunchArgs) = other ? other : k_mega_pixel<VARIANT, FMA, MEM, BIG>;
    LaunchArgs args = args_in;
    args.ap.tri_coop = MEM == PT_SCENE_SMEM;
    dim3 grid((args.W + 15) / 16, (args.nrows + 7) / 8), block(128);
    if (BIG && VARIANT == PT_VARIANT_GRID && !other) {
        // Warps of one CTA finish at different times and hold their registers until the last one does (ncu: 1.5 of ~8 warps
        // per scheduler wait at the final barrier).  Smaller CTAs return those slots earlier; PT_MEGA_WARPS = 1 | 2 | 4.
        static int nw = -1;
        if (nw == -1) { const char *e = getenv("PT_MEGA_WARPS"); nw = e ? atoi(e) : 4; if (nw != 1 && nw != 2) nw = 4; }
        if (nw == 2) { grid = dim3((args.W + 15) / 16, (args.nrows + 3) / 4); block = dim3(64); }
        if (nw == 1) { grid = dim3((args.W + 7) / 8, (args.nrows + 3) / 4); block = dim3(32); }
    }
    const size_t smem = MEM == PT_SCENE_SMEM ? (size_t)args.scene_bytes : 0;
    if (smem > 48 * 1024)
        PT_CUDA(cudaFuncSetAttribute(k_mega_pixel<VARIANT, FMA, MEM, BIG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                "opt-in shared memory");
    if (BIG) {
        static int order = -1;
        if (order == -1) { const char *e = getenv("PT_TILE_ORDER"); order = e ? atoi(e) : 1; }
        const size_t n = (size_t)grid.x * grid.y;
        // worth it when the launch is long (many samples) but only a few dozen waves short
        if (order && args.spp >= 16 && n >= (size_t)ctx->sm_count * 16) {
            TileOrderKey key;
            memset(&key, 0, sizeof(key));
            key.W = args.W; key.H = args.H; key.row_begin = args.row_begin; key.row_end = args.row_end; key.nrows = args.nrows;
            key.stripe_h = args.stripe_h; key.rank = args.rank; key.nranks = args.nranks; key.variant_fma = VARIANT * 4 + (FMA ? 2 : 0) + MEM + (other ? 64 : 0) + (int)block.x * 128;
            key.ntri = ctx->ntri_total; key.cam = args.cam;      // (not the scene version: a stale order is only a scheduling hint)
            for (int a = 0; a < 3; ++a) { key.bmin[a] = args.grid.bmin[a]; key.bmax[a] = args.grid.bmax[a]; key.cell[a] = args.grid.cell[a]; key.res[a] = args.grid.res[a]; }
            static_assert(sizeof(TileOrderKey) <= sizeof(ctx->tile_order_key), "tile order key buffer too small");
            if (ctx->tile_order_cap < n) {
                PT_CUDA(cudaStreamSynchronize(ctx->stream), "sync before growing the tile order");
                cudaFree(ctx->d_tile_order); cudaFree(ctx->d_cta_times);
                if (ctx->h_tile_order) cudaFreeHost(ctx->h_tile_order);
                if (ctx->h_cta_times) cudaFreeHost(ctx->h_cta_times);
                ctx->d_tile_order = nullptr; ctx->h_tile_order = nullptr; ctx->d_cta_times = nullptr; ctx->h_cta_times = nullptr;
                ctx->tile_order_cap = 0; ctx->tile_order_state = 0;
                PT_CUDA(cudaMalloc(&ctx->d_tile_order, n * 4), "alloc tile order");
                PT_CUDA(cudaMalloc(&ctx->d_cta_times, n * 16), "alloc CTA times");
                PT_CUDA(cudaMallocHost(&ctx->h_tile_order, n * 4), "alloc pinned tile order");
                PT_CUDA(cudaMallocHost(&ctx->h_cta_times, n * 16), "alloc pinned CTA times");
                ctx->tile_order_cap = n;
            }
            const bool same = ctx->tile_order_state != 0 && memcmp(&key, ctx->tile_order_key, sizeof(key)) == 0;
            if (!same) {
                // state 1: first launch of this geometry — raster order, every CTA records its span
                memcpy(ctx->tile_order_key, &key, sizeof(key));
                ctx->tile_order_state = 1;
                args.cta_times = ctx->d_cta_times;
            } else if (ctx->tile_order_state == 1) {
                // state 1 -> 2: the first launch recorded its CTA spans: sort the tiles by them, once
                if (tile_order_rebuild(ctx, n, true)) return 1;
                ctx->tile_order_state = 2;
            }
            if (ctx->tile_order_state == 2) {
                args.tile_order = ctx->d_tile_order;
                args.tiles_x = grid.x;
                grid = dim3((unsigned)n, 1);
            }
        }
        if (getenv("PT_CTA_TIMES")) {                 // diagnostics: pt_debug_read_scratch() returns the table (block-index order)
            const size_t nb = (size_t)grid.x * grid.y;
            if (pt_ensure_scratch(ctx, nb * 16 + 256)) return 1;
            unsigned long long *diag = (unsigned long long *)((char *)ctx->d_scratch + 256);
            if (!args.cta_times) { args.cta_times = diag; diag = nullptr; }
            kern<<<grid, block, smem, ctx->stream>>>(args);
            PT_CUDA(cudaGetLastError(), "launch k_mega_pixel");
            if (diag) PT_CUDA(cudaMemcpyAsync(diag, args.cta_times, nb * 16, cudaMemcpyDeviceToDevice, ctx->stream), "copy CTA times");
            return 0;
        }
    }
    kern<<<grid, block, smem, ctx->stream>>>(args);
    PT_CUDA(cudaGetLastError(), "launch k_mega_pixel");
    return 0;
}

template <int VARIANT, bool FMA, int MEM>
static int launch_pixel(pt_ctx ctx, const LaunchArgs &args) {
    if (VARIANT == PT_VARIANT_GRID ? ctx->ntri_total > 16384 : args.ap.ncl > 0) return launch_pixel_b<VARIANT, FMA, MEM, true>(ctx, args);
    return launch_pixel_b<VARIANT, FMA, MEM, false>(ctx, args);
}

template <bool FMA, int MEM>
static int launch_nodof(pt_ctx ctx, const LaunchArgs &args) {
    dim3 grid((args.W + 3) / 4, (args.nrows + 1) / 2), block(256);
    size_t smem = MEM == PT_SCENE_SMEM ? (size_t)args.scene_bytes : 0;
    k_mega_nodof<FMA, MEM><<<grid, block, smem, ctx->stream>>>(args);
    PT_CUDA(cudaGetLastError(), "launch k_mega_nodof");
    return 0;
}

template <bool FMA, int MEM>
static int launch_mega_am(pt_ctx ctx, int variant, const LaunchArgs &args) {
    switch (variant) {
        case PT_VARIANT_BASE: return launch_pixel<PT_VARIANT_BASE, FMA, MEM>(ctx, args);
        case PT_VARIANT_LMEM: return launch_pixel<PT_VARIANT_LMEM, FMA, MEM>(ctx, args);
        case PT_VARIANT_GRID: return launch_pixel<PT_VARIANT_GRID, FMA, MEM>(ctx, args);
        case PT_VARIANT_NODOF: return launch_nodof<FMA, MEM>(ctx, args);
    }
    return pt_fail(1, "unknown variant %d", variant);
}

}  // namespace pt

int pt_launch_mega(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args) {
    using namespace pt;
    const bool fma = p->arith != PT_ARITH_SEPARATE;
    if (p->scene_mem == PT_SCENE_SMEM)
        return fma ? launch_mega_am<true, PT_SCENE_SMEM>(ctx, p->variant, args)
                   : launch_mega_am<false, PT_SCENE_SMEM>(ctx, p->variant, args);
    int rc = pt_bind_const_scene(ctx, fma ? PT_ARITH_FMA : PT_ARITH_SEPARATE);
    if (rc) return rc;
    return fma ? launch_mega_am<true, PT_SCENE_CONST>(ctx, p->variant, args)
               : launch_mega_am<false, PT_SCENE_CONST>(ctx, p->variant, args);
}
